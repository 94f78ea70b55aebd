"""GPU suite: the fused observation front end (``ssd_frontend_forward``, csrc/frontend_b200.cu) over everything its C ABI
accepts, against the float64 restatement in ``frontend_ref.py``.

Bound, fixed per view before any run from the kernel header's own model (the tensor core's accumulation error grows linearly
with the MMAs chained on one TMEM accumulator, and 1e-6 holds at the 50 of V=15):

    |got - y64| <= tol(V) (1 + |y64|),    tol(V) = 1e-6 max(1, longest_chain(V) / 50)

Every check on random bytes or env observations also shows that the same inputs through the FC with its operands rounded to
tf32 (a kernel that lost its lo terms) miss that bound by at least 10x, so the bound can see such a bug.  Every case prints
its measured error as ``frontend-err <case> V=<v> err=<e> tol=<t> hi_only=<h>``.
"""
import ctypes as C
import types

import numpy as np
import pytest

import frontend_ref as R

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

DEV = "cuda:0"


def _weights(view, seed, conv_scale=1.0, fc_scale=1.0):
    """conv_w, conv_b, fc_w, fc_b as float32 numpy arrays (PyTorch's default init of the reference module)."""
    torch.manual_seed(seed)
    P = 2 * view - 1
    conv, fc = torch.nn.Conv2d(3, 6, 3, 1), torch.nn.Linear(6 * P * P, 32)
    w = [t.detach().numpy().astype(np.float32).copy() for t in (conv.weight, conv.bias, fc.weight, fc.bias)]
    w[0] *= np.float32(conv_scale)
    w[2] *= np.float32(fc_scale)
    return w


def _front_end(w, view, slope=0.01):
    from homophily_marl_b200.frontend import ObsFrontEnd
    return ObsFrontEnd(*w, view, negative_slope=slope, device=DEV)


def _random_buf(n, seed):
    return np.random.RandomState(seed).randint(0, 256, size=n).astype(np.uint8)


def _expect(case, view, got, host, rows, lay, w, slope, hi_check=True, scale="y"):
    """Asserts the bound on `got` (numpy [rows, 32]) and, with hi_check, that the hi-only FC misses it by >= 10x.

    scale="M" measures the error against 1 + M, M = |fc_b| + sum |W||a| the condition scale of the FC sum, instead of
    1 + |y|: with trained-like weights the sum cancels (M / (1 + |y|) reaches ~1 000 at 16x the default init) and no fp32
    contraction meets the 1 + |y| form there -- torch's own fp32 matmul of the exact activations measures 2.2e-5."""
    slope = float(np.float32(slope))                          # the kernel's slope is the float32 one
    y, M = R.forward64(host, rows, lay["AS"], lay["PS"], lay["RP"], view, *w, slope)
    tol = R.tolerance(view)

    def rel(v):
        return float((np.abs(np.asarray(v, np.float64) - y) / (1 + (M if scale == "M" else np.abs(y)))).max()) if y.size else 0.0
    err = rel(got)
    herr = rel(R.forward64_hi_only(host, rows, lay["AS"], lay["PS"], lay["RP"], view, *w, slope)) if hi_check else float("nan")
    print(f"frontend-err {case} V={view} err={err:.3e} tol={tol:.2e} hi_only={herr:.3e}"
          + (f" scale=1+M (vs 1+|y|: {R.rel_err(got, y):.3e})" if scale == "M" else ""))
    assert np.isfinite(got).all(), case
    assert err <= tol, (case, view, err, tol)
    if hi_check:
        assert herr >= 10 * tol, (case, view, herr, tol)
    return y


def _run(fe, host, rows, lay, offset=0, out=None):
    buf = torch.as_tensor(host).to(DEV)
    got = fe.forward(buf[offset:] if offset else buf, rows, lay["AS"], lay["PS"], lay["RP"], out=out)
    torch.cuda.synchronize()
    return got


def _used_bytes(size, rows, lay, view):
    """Mask of the bytes the module reads (pixel (c, y, x) of every row, x, y < N); everything else is padding."""
    N = 2 * view + 1
    r, c, y, x = np.meshgrid(np.arange(rows), np.arange(3), np.arange(N), np.arange(N), indexing="ij")
    used = np.zeros(size, dtype=bool)
    used[(r * lay["AS"] + c * lay["PS"] + y * lay["RP"] + x).ravel()] = True
    return used


def _auto_grid(view, rows):
    """The grid ssd_frontend_forward picks without SSD_B200_FRONTEND_GRID (restated), and the number of (tile, chunk) units."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    P = 2 * view - 1
    n_chunks, tiles = P * ((P + 15) // 16), -(-rows // 128)
    units = tiles * n_chunks
    grid = min(units, sms)
    share = units / grid
    best = share + 1.5 * (2.0 if share < n_chunks else float(int(share / n_chunks) + 2))
    for s in range(1, n_chunks + 1):
        if tiles * s > sms:
            break
        cost = (n_chunks + s - 1) // s + 1.5
        if cost < best - 1e-9:
            best, grid = cost, tiles * s
    return grid, units


# ---------------------------------------------------------------------------------------------------- numeric contract

@pytest.mark.parametrize("view", range(1, 32))
def test_every_view_with_a_partial_last_tile(view):
    rows, lay = 3 * 128 + 5, R.env_layout(view)
    w = _weights(view, seed=view)
    host = _random_buf(rows * lay["AS"], seed=view)          # pad bytes are garbage too
    fe = _front_end(w, view)
    _expect("views", view, _run(fe, host, rows, lay).cpu().numpy(), host, rows, lay, w, 0.01)
    fe.close()


@pytest.mark.parametrize("view", [1, 7, 15, 31])
@pytest.mark.parametrize("slope", [0.0, 0.2, 1.0])
def test_slopes_with_both_branches_taken(view, slope):
    rows, lay = 3 * 128 + 5, R.env_layout(view)
    w = _weights(view, seed=100 + view)
    host = _random_buf(rows * lay["AS"], seed=200 + view)
    P = 2 * view - 1
    pre = R.features64(host, rows, lay["AS"], lay["PS"], lay["RP"], view, w[0], np.zeros(6, np.float32), 1.0).reshape(rows, 6, P * P)
    w[1] = (-np.median(pre.transpose(1, 0, 2).reshape(6, -1), axis=1) + w[1] * 0.1).astype(np.float32)   # about half negative
    conv_neg = (R.features64(host, rows, lay["AS"], lay["PS"], lay["RP"], view, w[0], w[1], 1.0) < 0).mean()
    assert 0.2 <= conv_neg <= 0.8, conv_neg
    fe = _front_end(w, view, slope)
    y = _expect(f"slope{slope}", view, _run(fe, host, rows, lay).cpu().numpy(), host, rows, lay, w, slope)
    fc_neg = (y < 0).mean() if slope > 0 else (y == 0).mean()
    assert 0.05 <= fc_neg <= 0.95, fc_neg                     # the epilogue's LeakyReLU sees both signs too
    fe.close()


def _max_lo(w):
    """Moves every weight to just below the tie between two tf32 values: the largest lo = w - rn_tf32(w) there is."""
    bits = np.asarray(w, dtype=np.float32).view(np.uint32)
    return ((bits & np.uint32(0xFFFFE000)) | np.uint32(0x0FFF)).view(np.float32)


@pytest.mark.parametrize("view", [7, 15])
@pytest.mark.parametrize("regime", ["default", "x16", "fc_exact_tf32", "fc_max_lo"])
def test_weight_regimes(view, regime):
    rows, lay = 3 * 128 + 5, R.env_layout(view)
    w = _weights(view, seed=300 + view, **(dict(conv_scale=16.0, fc_scale=16.0) if regime == "x16" else {}))
    if regime == "fc_exact_tf32":
        w[2] = R.tf32_rna(w[2])
        assert np.array_equal(R.tf32_rna(w[2]), w[2])
    elif regime == "fc_max_lo":
        w[2] = _max_lo(w[2])
        lo = w[2].astype(np.float64) - R.tf32_rna(w[2]).astype(np.float64)
        assert (np.abs(lo) == 4095 * np.spacing(np.abs(w[2]))).all()             # 4095 of the 8192 fp32 ulps under a tf32 one
    host = _random_buf(rows * lay["AS"], seed=400 + view)
    fe = _front_end(w, view)
    _expect(regime, view, _run(fe, host, rows, lay).cpu().numpy(), host, rows, lay, w, 0.01, scale="M" if regime == "x16" else "y")
    fe.close()


@pytest.mark.parametrize("view", [7, 15, 31])
@pytest.mark.parametrize("fill", [0, 255])
def test_constant_inputs(view, fill):
    rows, lay = 3 * 128 + 5, R.env_layout(view)
    w = _weights(view, seed=500 + view)
    host = np.full(rows * lay["AS"], fill, dtype=np.uint8)
    fe = _front_end(w, view)
    got = _run(fe, host, rows, lay)
    _expect(f"fill{fill}", view, got.cpu().numpy(), host, rows, lay, w, 0.01, hi_check=False)
    for t in range(0, rows, 128):                             # one tile: the same operations on the same values
        tile = got[t:t + 128]
        assert torch.equal(tile, tile[:1].expand_as(tile)), t
    assert ((got - got[:1]).abs() / (1 + got[:1].abs())).max().item() <= R.tolerance(view)   # tiles: fp32 summation order
    fe.close()


@pytest.mark.parametrize("name,mp,n,view", [("cleanup", "default5", 5, 7), ("harvest", "default5", 5, 15)])
def test_env_observations(name, mp, n, view):
    from homophily_marl_b200.batch_env import SSDBatchEnv
    B = 100
    env = SSDBatchEnv(name, B, n, map=mp, view_size=view, seed=9, extra_args=dict(random_spawn_point=True, random_spawn_rotation=None))
    env.reset()
    rs = np.random.RandomState(2)
    for _ in range(7):
        env.step(torch.as_tensor(rs.randint(0, env.n_actions, size=(B, n)).astype(np.uint8), device=env.device))
    torch.cuda.synchronize()
    lay = dict(AS=env.layout.obs_agent_stride, PS=env.layout.obs_plane_stride, RP=env.layout.obs_row_stride)
    host = env.obs_buf.view(-1).cpu().numpy()
    w = _weights(view, seed=600 + view)
    fe = _front_end(w, view)
    _expect(f"env-{name}", view, fe.forward_env(env).cpu().numpy(), host, B * n, lay, w, 0.01)
    fe.close()
    env.close()


def _layout(view, kind):
    N = 2 * view + 1
    lay = R.env_layout(view)
    if kind in ("rp+4", "rp+60"):
        RP = lay["RP"] + int(kind[3:])
        lay = dict(RP=RP, PS=N * RP, AS=(3 * N * RP + 15) // 16 * 16)
    elif kind == "ps+12":
        lay = dict(lay, PS=N * lay["RP"] + 12, AS=(3 * (N * lay["RP"] + 12) + 15) // 16 * 16)
    elif kind == "as+4":
        lay = dict(lay, AS=3 * lay["PS"] + 4)
    return lay


@pytest.mark.parametrize("view", [7, 9, 15])
@pytest.mark.parametrize("kind", ["rp+4", "rp+60", "ps+12", "as+4", "offset4"])
def test_layouts_beyond_the_envs(view, kind):
    rows, lay = 3 * 128 + 5, _layout(view, kind)
    off = 4 if kind == "offset4" else 0
    w = _weights(view, seed=700 + view)
    host = _random_buf(rows * lay["AS"] + off, seed=800 + view)
    fe = _front_end(w, view)
    got = _run(fe, host, rows, lay, offset=off).cpu().numpy()
    _expect(kind, view, got, host[off:], rows, lay, w, 0.01)
    fe.close()


# ---------------------------------------------------------------------------------------------------- bit-exact invariances

@pytest.mark.parametrize("view,kind", [(7, "env"), (15, "env"), (9, "as+4"), (15, "rp+60")])
def test_pads_and_other_rows_do_not_reach_a_rows_output(view, kind):
    rows = 3 * 128 + 5
    lay = R.env_layout(view) if kind == "env" else _layout(view, kind)
    w = _weights(view, seed=900 + view)
    host = _random_buf(rows * lay["AS"], seed=1000 + view)
    fe = _front_end(w, view)
    ref = _run(fe, host, rows, lay).clone()
    used = _used_bytes(host.size, rows, lay, view)
    assert (~used).any()
    pads = host.copy()
    pads[~used] = host[~used] ^ (_random_buf(int((~used).sum()), seed=1) | 1)      # every pad byte changes
    assert torch.equal(_run(fe, pads, rows, lay), ref)        # pad pixels only ever meet zero FC weights
    odd = host.copy().reshape(rows, lay["AS"])
    odd[1::2] = _random_buf(odd[1::2].size, seed=2).reshape(odd[1::2].shape)
    got = _run(fe, odd.reshape(-1), rows, lay)
    assert torch.equal(got[0::2], ref[0::2])                  # tensor-core rows are independent
    assert not torch.equal(got[1::2], ref[1::2])
    fe.close()


def test_out_rows_beyond_rows_stay_untouched():
    view, rows = 15, 3 * 128 + 5
    lay = R.env_layout(view)
    w = _weights(view, seed=11)
    host = _random_buf(rows * lay["AS"], seed=12)
    fe = _front_end(w, view)
    big = torch.full((rows + 8, 32), float("nan"), device=DEV)
    got = _run(fe, host, rows, lay, out=big[:rows])
    assert got.data_ptr() == big.data_ptr()
    assert torch.isnan(big[rows:]).all() and not torch.isnan(big[:rows]).any()
    _expect("out-bounds", view, big[:rows].cpu().numpy(), host, rows, lay, w, 0.01)
    fe.close()


# ---------------------------------------------------------------------------------------------------- work division

@pytest.mark.parametrize("view,rows", [(7, 2560), (15, 300), (31, 200), (3, 200)])
def test_every_grid_gives_the_bound_and_repeats_bit_for_bit(view, rows, monkeypatch):
    lay = R.env_layout(view)
    w = _weights(view, seed=1100 + view)
    host = _random_buf(rows * lay["AS"], seed=1200 + view)
    auto, units = _auto_grid(view, rows)
    if (view, rows) == (7, 2560) and torch.cuda.get_device_properties(0).multi_processor_count == 148:
        assert auto == 140                                    # an env range of the batched runner: 7 CTAs per 13-chunk tile
    grids = [1, 2, 3, 7, 13, 64, None] + ([units] if units <= auto else [])
    fe = _front_end(w, view)
    y = _expect("grid-auto", view, _run(fe, host, rows, lay).cpu().numpy(), host, rows, lay, w, 0.01)
    for g in grids:
        if g is None:
            monkeypatch.delenv("SSD_B200_FRONTEND_GRID", raising=False)
        else:
            monkeypatch.setenv("SSD_B200_FRONTEND_GRID", str(g))
        a = _run(fe, host, rows, lay).clone()
        b = _run(fe, host, rows, lay)
        assert torch.equal(a, b), g
        err = R.rel_err(a.cpu().numpy(), y)
        print(f"frontend-err grid{g or auto} V={view} err={err:.3e} tol={R.tolerance(view):.2e}")
        assert err <= R.tolerance(view), (g, err)
    fe.close()


def test_growing_batches_and_changing_grids_on_one_handle(monkeypatch):
    """The handle allocates tile counters in blocks of 1 024 tiles: 131 200 rows (1 025 tiles) re-allocate them.  Each call
    must find the counters and scratch its predecessors used, at other grids and tile counts, left clean."""
    view = 3
    lay = R.env_layout(view)
    w = _weights(view, seed=13)
    fe = _front_end(w, view)
    seq = [(300, "1"), (300, None), (20480, "64"), (20480, None), (131200, "97"), (131200, None), (300, "7"), (20480, "2"), (300, "13")]
    for i, (rows, grid) in enumerate(seq):
        if grid is None:
            monkeypatch.delenv("SSD_B200_FRONTEND_GRID", raising=False)
        else:
            monkeypatch.setenv("SSD_B200_FRONTEND_GRID", grid)
        host = _random_buf(rows * lay["AS"], seed=1300 + i)
        _expect(f"sequence{i}-rows{rows}-grid{grid or 'auto'}", view, _run(fe, host, rows, lay).cpu().numpy(), host, rows, lay, w, 0.01,
                hi_check=rows == 300)
    fe.close()


# ---------------------------------------------------------------------------------------------------- argument validation

def test_forward_rejects_bad_strides_and_pointers_without_a_launch():
    from homophily_marl_b200 import _capi
    view, rows = 7, 130
    N, lay = 15, R.env_layout(7)
    w = _weights(view, seed=14)
    fe = _front_end(w, view)
    lib = fe.lib
    buf = torch.zeros(rows * lay["AS"] + 64, dtype=torch.uint8, device=DEV)
    out = torch.full((rows + 4, 32), float("nan"), device=DEV)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    before = lib.ssd_frontend_last_cuda_error()

    def fwd(obs_ptr=None, n=rows, AS=lay["AS"], PS=lay["PS"], RP=lay["RP"], out_ptr=None, h=fe._h):
        return lib.ssd_frontend_forward(h, obs_ptr or buf.data_ptr(), n, AS, PS, RP, out_ptr or out.data_ptr(), stream)

    bad = [dict(RP=12), dict(RP=N), dict(RP=lay["RP"] + 2), dict(PS=N * lay["RP"] - 4), dict(PS=N * lay["RP"] + 2),
           dict(AS=3 * lay["PS"] - 4), dict(AS=3 * lay["PS"] + 2), dict(obs_ptr=buf.data_ptr() + 1), dict(out_ptr=out.data_ptr() + 4),
           dict(n=-1)]
    for kw in bad:
        assert fwd(**kw) == _capi.SSD_ERR_INVALID, kw
    w31 = _weights(31, seed=15)
    fe31 = _front_end(w31, 31)
    tiles = (1 << 31) // 244 + 1                              # V=31: 244 chunks per tile, units = tiles * 244 >= 2^31
    assert (tiles - 1) * 244 < (1 << 31) <= tiles * 244
    assert fwd(n=tiles * 128, AS=R.env_layout(31)["AS"], PS=R.env_layout(31)["PS"], RP=R.env_layout(31)["RP"], h=fe31._h) == _capi.SSD_ERR_INVALID
    torch.cuda.synchronize()
    assert torch.isnan(out).all()                             # nothing was launched
    assert lib.ssd_frontend_last_cuda_error() == before
    assert fwd() == _capi.SSD_OK                              # the same arguments with good strides do launch
    torch.cuda.synchronize()
    assert not torch.isnan(out[:rows]).any() and torch.isnan(out[rows:]).all()
    empty = fe.forward(buf, 0, lay["AS"], lay["PS"], lay["RP"])
    assert empty.shape == (0, 32) and empty.dtype == torch.float32 and empty.is_cuda
    fe31.close()
    fe.close()


def test_forward_rejects_an_out_it_cannot_write():
    view, rows = 7, 130
    lay = R.env_layout(view)
    fe = _front_end(_weights(view, seed=16), view)
    buf = torch.zeros(rows * lay["AS"], dtype=torch.uint8, device=DEV)
    bad = [torch.empty((rows, 32), dtype=torch.float16, device=DEV), torch.empty((rows, 31), device=DEV),
           torch.empty((rows - 1, 32), device=DEV), torch.empty((rows * 32,), device=DEV),
           torch.empty((32, rows), device=DEV).t(), torch.empty((rows, 64), device=DEV)[:, :32], torch.empty((rows, 32))]
    for out in bad:
        with pytest.raises(ValueError):
            fe.forward(buf, rows, lay["AS"], lay["PS"], lay["RP"], out=out)
    with pytest.raises(ValueError):
        fe.forward(buf.cpu(), rows, lay["AS"], lay["PS"], lay["RP"])
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            fe.forward(buf.to("cuda:1"), rows, lay["AS"], lay["PS"], lay["RP"])
        with pytest.raises(ValueError):
            fe.forward(buf, rows, lay["AS"], lay["PS"], lay["RP"], out=torch.empty((rows, 32), device="cuda:1"))
    fe.close()


# ---------------------------------------------------------------------------------------------------- concurrency

def test_two_handles_on_two_streams_without_a_host_sync():
    view, rows = 7, 2560
    lay = R.env_layout(view)
    ws = [_weights(view, seed=17 + i) for i in range(2)]
    hosts = [_random_buf(rows * lay["AS"], seed=1400 + i) for i in range(2)]
    fes = [_front_end(w, view) for w in ws]
    bufs = [torch.as_tensor(h).to(DEV) for h in hosts]
    outs = [torch.empty((rows, 32), device=DEV) for _ in range(2)]
    torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=DEV) for _ in range(2)]
    for fe, buf, out, s in zip(fes, bufs, outs, streams):
        with torch.cuda.stream(s):
            fe.forward(buf, rows, lay["AS"], lay["PS"], lay["RP"], out=out)
    torch.cuda.synchronize()
    for i in range(2):
        _expect(f"two-streams{i}", view, outs[i].cpu().numpy(), hosts[i], rows, lay, ws[i], 0.01)
    for fe in fes:
        fe.close()


def test_batched_runner_ranges_each_use_their_own_handle(monkeypatch):
    """env_groups = 4 with the fused front end: every range's features equal fp64 on exactly the rows the runner stored."""
    from homophily_marl_b200.batched_runner import BatchedEpisodeRunner
    from homophily_marl_b200.frontend import MacFrontEnd, ObsFrontEnd
    from test_batched_runner import FakeBatch, _scheme
    B, T, n, view, G = 128, 20, 3, 7, 4
    N = 2 * view + 1
    extra = dict(random_spawn_point=True, random_spawn_rotation=None, disable_rotation_action=False,
                 disable_fire_action=False, obs_color="full")
    env_args = dict(num_agents=n, render=False, episode_limit=T, is_replay=False, view_size=view, map="default3", extra_args=extra, seed=5)
    args = types.SimpleNamespace(batch_size_run=B, env="cleanup", env_args=env_args, device=DEV, name="homophily", mac="homophily_mac",
                                 n_actions=None, ind_reward=True, runner_log_interval=10 ** 9, test_nepisode=B, env_groups=G)
    runner = BatchedEpisodeRunner(args, types.SimpleNamespace(log_stat=lambda k, v, t: None))
    info = runner.get_env_info()
    A = args.n_actions = info["n_actions"]
    g = torch.Generator().manual_seed(3)
    table = torch.randint(0, A, (B, T + 1, n, 1), generator=g).to(DEV)
    table_inc = torch.randint(0, 3, (B, T + 1, n, n, 1), generator=g).to(DEV)
    runner.use_batch_factory(lambda: FakeBatch(_scheme(n, A, *info["state_dims"], N), B, T + 1, DEV))

    torch.manual_seed(19)
    P = 2 * view - 1
    module = torch.nn.Sequential(torch.nn.Conv2d(3, 6, 3, 1), torch.nn.LeakyReLU(), torch.nn.Flatten(),
                                 torch.nn.Linear(6 * P * P, 32), torch.nn.LeakyReLU()).to(DEV)

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

    records = []
    forward = ObsFrontEnd.forward

    def recording(self, obs_buf, rows, agent_stride, plane_stride, row_stride, out=None):
        got = forward(self, obs_buf, rows, agent_stride, plane_stride, row_stride, out=out)
        records.append((self, obs_buf[:rows * agent_stride].clone(), got.clone(), rows, agent_stride, plane_stride, row_stride))
        return got                                            # the clones run on the current (the range's) stream

    monkeypatch.setattr(ObsFrontEnd, "forward", recording)
    runner.mac = MAC()
    runner.front = MacFrontEnd(runner.mac, runner.env)
    batch = runner.run(test_mode=True)
    torch.cuda.synchronize()
    assert len(records) == (T + 1) * G                        # t-major, range-minor: call i is range i % G at step i // G

    w = [t.detach().float().cpu().numpy() for t in (module[0].weight, module[0].bias, module[3].weight, module[3].bias)]
    Bg = B // G
    errs, herrs, tol = [], [], R.tolerance(view)
    for i, (_, obs, got, rows, AS, PS, RP) in enumerate(records):
        t, k = divmod(i, G)
        assert rows == Bg * n
        stored = (batch["obs"][k * Bg:(k + 1) * Bg, t] * 256).to(torch.uint8).reshape(rows, 3, N, N)
        assert torch.equal(obs.as_strided((rows, 3, N, N), (AS, PS, RP, 1)), stored), (t, k)
        host = obs.cpu().numpy()
        y, _ = R.forward64(host, rows, AS, PS, RP, view, *w, float(np.float32(0.01)))
        errs.append(R.rel_err(got.cpu().numpy(), y))
        herrs.append(R.rel_err(R.forward64_hi_only(host, rows, AS, PS, RP, view, *w, float(np.float32(0.01))), y))
    print(f"frontend-err runner V={view} err={max(errs):.3e} tol={tol:.2e} hi_only={min(herrs):.3e}")
    assert max(errs) <= tol, [(i, e) for i, e in enumerate(errs) if e > tol][:8]
    assert min(herrs) >= 10 * tol
    handles = [{id(rec[0]) for rec in records[k::G]} for k in range(G)]
    assert all(len(h) == 1 for h in handles) and len(set.union(*handles)) == G, "env ranges must not share a front-end handle"
    runner.front.detach()
    runner.close_env()
