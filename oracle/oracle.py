"""TEST INFRASTRUCTURE ONLY -- ctypes wrapper around ``libssd_oracle.so``
(the plain-C restatement in ``ssd_oracle.c``).  Imported by ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline / ``--impl reference``
legs only; never by ``homophily_marl_b200``.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libssd_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    """Compile the C restatement with gcc (OpenMP when the toolchain has it).  In a read-only tree the library is built
    once per source version into a per-user cache in the temporary directory; returns the path of the library."""
    src = os.path.join(HERE, "ssd_oracle.c")
    hdr = os.path.join(HERE, "ssd_oracle.h")
    if not force and os.path.exists(LIB_PATH) and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(src), os.path.getmtime(hdr)):
        return LIB_PATH
    out = LIB_PATH
    if not os.access(HERE, os.W_OK):                          # one cached library per source version and user
        h = hashlib.sha256(b"".join(open(f, "rb").read() for f in (src, hdr))).hexdigest()[:16]
        out = os.path.join(tempfile.gettempdir(), f"ssd_oracle_{os.getuid()}", f"libssd_oracle_{h}.so")
        if os.path.exists(out) and not force:
            return out
        os.makedirs(os.path.dirname(out), exist_ok=True)
    tmp = f"{out}.{os.getpid()}.tmp"
    base = ["-O2", "-ffp-contract=off", "-fPIC", "-std=c11", "-shared", "-o", tmp, src, "-lm"]
    errors = []
    for cc in ("/usr/bin/gcc", shutil.which("gcc"), os.environ.get("CC"), shutil.which("cc")):
        if not cc or not os.path.exists(cc):
            continue
        for omp in (["-fopenmp"], []):
            r = subprocess.run([cc] + omp + base, capture_output=True, text=True)
            if r.returncode == 0:
                os.replace(tmp, out)                          # atomic: concurrent processes never load a partial file
                return out
            errors.append(r.stderr[-300:])
    raise RuntimeError("could not build the oracle: " + " | ".join(errors))


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.ssdo_sizeof_map.restype = C.c_ulong
        L.ssdo_sizeof_env.restype = C.c_ulong
        L.ssdo_map_init.restype = C.c_int
        L.ssdo_map_init.argtypes = [C.c_void_p, C.c_int, C.c_char_p] + [C.c_int] * 6 + [C.c_double] * 4 + [C.c_void_p, C.c_int, C.c_int]
        L.ssdo_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32]
        L.ssdo_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 4
        L.ssdo_render_obs.argtypes = [C.c_void_p] * 3
        L.ssdo_render_state.argtypes = [C.c_void_p] * 3
        L.ssdo_batch_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_int]
        L.ssdo_batch_step.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint64, C.c_uint32] + [C.c_void_p] * 5 + [C.c_int]
        L.ssdo_philox4x32_10.argtypes = [C.c_void_p] * 3
        _lib = L
    return _lib


MAX_CELLS, MAX_AGENTS = 2048, 16
ENV_DTYPE = np.dtype([("grid", np.uint8, MAX_CELLS), ("pos", np.int32, MAX_AGENTS),
                      ("orient", np.uint8, MAX_AGENTS), ("ep_ret", np.int32, MAX_AGENTS),
                      ("t", np.int32), ("tick", np.uint32), ("error", np.int32)], align=True)


class _Draws(C.Structure):
    _fields_ = [(k, C.c_void_p) for k in ("prio", "u_apple", "u_waste", "wkey", "spawn_key", "rot")]


def philox(ctr, key):
    out = np.zeros(4, dtype=np.uint32)
    c = np.asarray(ctr, dtype=np.uint32)
    k = np.asarray(key, dtype=np.uint32)
    lib().ssdo_philox4x32_10(c.ctypes.data, k.ctypes.data, out.ctypes.data)
    return out


def _ptr(a):
    return None if a is None else a.ctypes.data


class OracleBatch:
    """B independent oracle envs sharing one map."""

    def __init__(self, kind, rows, n_agents, view, episode_limit, full_color,
                 threshold_depletion=0.0, threshold_restoration=0.0, waste_spawn_prob=0.0,
                 apple_respawn_prob=0.0, spawn_prob=(0, 0, 0, 0), fire_cost=1, hit_penalty=0,
                 n_envs=1, seed=0, env_gid0=0, random_spawn_point=False, spawn_rotation=0):
        L = lib()
        assert L.ssdo_sizeof_env() == ENV_DTYPE.itemsize, (L.ssdo_sizeof_env(), ENV_DTYPE.itemsize)
        self.H, self.W = len(rows), len(rows[0])
        self.G, self.n, self.V, self.N = self.H * self.W, n_agents, view, 2 * view + 1
        self.B, self.seed, self.gid0 = n_envs, seed, env_gid0
        self.random_spawn_point = bool(random_spawn_point)
        self.spawn_rotation = -1 if spawn_rotation is None else int(spawn_rotation)
        self._map = np.zeros(L.ssdo_sizeof_map(), dtype=np.uint8)
        sp = np.asarray(spawn_prob, dtype=np.float64)
        rc = L.ssdo_map_init(self._map.ctypes.data, kind, "".join(rows).encode(), self.H, self.W, n_agents, view,
                             episode_limit, int(full_color), threshold_depletion, threshold_restoration,
                             waste_spawn_prob, apple_respawn_prob, sp.ctypes.data, fire_cost, hit_penalty)
        if rc != 0:
            raise ValueError("ssdo_map_init failed: %d" % rc)
        self.envs = np.zeros(n_envs, dtype=ENV_DTYPE)

    @classmethod
    def from_spec(cls, spec, **kw):
        p = spec.params
        return cls(spec.kind, spec.rows, spec.n_agents, spec.view, spec.episode_limit, spec.obs_color == "full",
                   p.threshold_depletion, p.threshold_restoration, p.waste_spawn_prob, p.apple_respawn_prob,
                   p.spawn_prob, spec.fire_cost, spec.hit_penalty, **kw)

    # ---- state views ---------------------------------------------------
    @property
    def grid(self):
        return self.envs["grid"][:, :self.G].reshape(self.B, self.H, self.W)

    @property
    def pos(self):       # cell index [B, n]
        return self.envs["pos"][:, :self.n]

    @property
    def pos_rc(self):
        p = self.pos
        return np.stack([p // self.W, p % self.W], axis=-1)

    @property
    def orient(self):
        return self.envs["orient"][:, :self.n]

    @property
    def ep_ret(self):
        return self.envs["ep_ret"][:, :self.n]

    def set_state(self, b, grid=None, pos_rc=None, orient=None):
        if grid is not None:
            self.envs["grid"][b, :self.G] = np.asarray(grid, dtype=np.uint8).reshape(-1)
        if pos_rc is not None:
            pr = np.asarray(pos_rc)
            self.envs["pos"][b, :self.n] = pr[:, 0] * self.W + pr[:, 1]
        if orient is not None:
            self.envs["orient"][b, :self.n] = orient

    # ---- single-env entry points with optional injected draws ----------------
    def _draws(self, d):
        if d is None:
            return None, None
        keep = {k: (None if d.get(k) is None else np.ascontiguousarray(d[k], dtype=np.uint8 if k == "rot" else np.uint32))
                for k in ("prio", "u_apple", "u_waste", "wkey", "spawn_key", "rot")}
        s = _Draws(**{k: _ptr(v) for k, v in keep.items()})
        return s, keep

    def reset_one(self, b=0, draws=None):
        s, keep = self._draws(draws)
        lib().ssdo_reset(self._map.ctypes.data, self.envs[b:b + 1].ctypes.data, int(self.random_spawn_point),
                         self.spawn_rotation, C.byref(s) if s is not None else None, self.seed, self.gid0 + b)

    def step_one(self, actions, b=0, draws=None):
        s, keep = self._draws(draws)
        a = np.ascontiguousarray(actions, dtype=np.uint8)
        reward = np.zeros(self.n, dtype=np.int8)
        clean = np.zeros(self.n, dtype=np.uint8)
        cnt = np.zeros(1, dtype=np.uint16)
        done = np.zeros(1, dtype=np.uint8)
        lib().ssdo_step(self._map.ctypes.data, self.envs[b:b + 1].ctypes.data, a.ctypes.data,
                        C.byref(s) if s is not None else None, self.seed, self.gid0 + b,
                        reward.ctypes.data, clean.ctypes.data, cnt.ctypes.data, done.ctypes.data)
        return reward, clean, int(cnt[0]), bool(done[0])

    def obs_one(self, b=0):
        out = np.zeros((self.n, 3, self.N, self.N), dtype=np.uint8)
        lib().ssdo_render_obs(self._map.ctypes.data, self.envs[b:b + 1].ctypes.data, out.ctypes.data)
        return out

    def state_one(self, b=0):
        out = np.zeros((3, self.H, self.W), dtype=np.uint8)
        lib().ssdo_render_state(self._map.ctypes.data, self.envs[b:b + 1].ctypes.data, out.ctypes.data)
        return out

    # ---- batch entry points (Philox draws) ------------------------------------
    def reset(self, threads=1):
        lib().ssdo_batch_reset(self._map.ctypes.data, self.envs.ctypes.data, self.B, int(self.random_spawn_point),
                               self.spawn_rotation, self.seed, self.gid0, threads)

    def step(self, actions, want_obs=True, threads=1, out=None):
        a = np.ascontiguousarray(actions, dtype=np.uint8).reshape(self.B, self.n)
        if out is None:
            out = dict(reward=np.zeros((self.B, self.n), np.int8), clean=np.zeros((self.B, self.n), np.uint8),
                       apple_cnt=np.zeros(self.B, np.uint16), done=np.zeros(self.B, np.uint8),
                       obs=np.zeros((self.B, self.n, 3, self.N, self.N), np.uint8) if want_obs else None)
        lib().ssdo_batch_step(self._map.ctypes.data, self.envs.ctypes.data, self.B, a.ctypes.data, self.seed, self.gid0,
                              out["reward"].ctypes.data, out["clean"].ctypes.data, out["apple_cnt"].ctypes.data,
                              out["done"].ctypes.data, _ptr(out["obs"]) if want_obs else None, threads)
        return out
