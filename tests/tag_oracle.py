"""TEST INFRASTRUCTURE ONLY -- ``OracleBatch`` with tagging-out timers: a ctypes wrapper around ``tests/tag_oracle.c``.

``TagOracleBatch`` takes every argument ``OracleBatch`` takes plus ``tag_timeout`` (from ``spec.tag_timeout`` in
``from_spec``), keeps the timers in ``tag_out`` ([B, n] u8, 0 = in play) and runs the tagging spec of DESIGN.md §3 item 11.
With ``tag_timeout`` 0 and no timer set it computes what ``OracleBatch`` computes (tests/test_oracle_tagging.py checks that).
The library is built once per source version into a per-user cache in the temporary directory.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
_lib = None


def build() -> str:
    srcs = [os.path.join(HERE, "tag_oracle.c"), os.path.join(ORACLE_DIR, "ssd_oracle.c"), os.path.join(ORACLE_DIR, "ssd_oracle.h")]
    h = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"ssd_oracle_{os.getuid()}", f"libssd_tag_oracle_{h}.so")
    if os.path.exists(out):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    tmp = f"{out}.{os.getpid()}.tmp"
    base = ["-O2", "-ffp-contract=off", "-fPIC", "-std=c11", "-shared", "-I", ORACLE_DIR, "-o", tmp, srcs[0], "-lm"]
    errors = []
    for cc in ("/usr/bin/gcc", shutil.which("gcc"), os.environ.get("CC"), shutil.which("cc")):
        if not cc or not os.path.exists(cc):
            continue
        for omp in (["-fopenmp"], []):
            r = subprocess.run([cc] + omp + base, capture_output=True, text=True)
            if r.returncode == 0:
                os.replace(tmp, out)
                return out
            errors.append(r.stderr[-300:])
    raise RuntimeError("could not build the tagging reference: " + " | ".join(errors))


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        P, I = C.c_void_p, C.c_int
        L.ssdt_submaps.argtypes = [P, P]
        L.ssdt_step.argtypes = [P, P, P, P, P, P, C.c_uint64, C.c_uint32, I, I, I, P, P, P, P]
        L.ssdt_render_obs.argtypes = [P, P, P, P]
        L.ssdt_render_state.argtypes = [P, P, P, P]
        L.ssdt_batch_step.argtypes = [P, P, P, P, I, P, C.c_uint64, C.c_uint32, I, I, I, P, P, P, P, P, I]
        _lib = L
    return _lib


class TagOracleBatch(O.OracleBatch):
    def __init__(self, *args, tag_timeout=0, **kw):
        super().__init__(*args, **kw)
        self.tag_timeout = int(tag_timeout)
        self._tag = np.zeros((self.B, O.MAX_AGENTS), dtype=np.uint8)
        self._subs = np.zeros((self.n + 1) * O.lib().ssdo_sizeof_map(), dtype=np.uint8)
        lib().ssdt_submaps(self._map.ctypes.data, self._subs.ctypes.data)

    @classmethod
    def from_spec(cls, spec, **kw):
        kw.setdefault("tag_timeout", spec.tag_timeout)
        return super().from_spec(spec, **kw)

    @property
    def tag_out(self):   # [B, n] steps each agent is still out of play; 0 = on the map
        return self._tag[:, :self.n]

    def set_state(self, b, grid=None, pos_rc=None, orient=None, tag_out=None):
        super().set_state(b, grid=grid, pos_rc=pos_rc, orient=orient)
        if tag_out is not None:
            self._tag[b, :self.n] = tag_out

    def reset_one(self, b=0, draws=None):
        super().reset_one(b, draws)
        self._tag[b] = 0

    def reset(self, threads=1):
        super().reset(threads)
        self._tag[:] = 0

    def step_one(self, actions, b=0, draws=None):
        s, keep = self._draws(draws)
        a = np.ascontiguousarray(actions, dtype=np.uint8)
        reward = np.zeros(self.n, dtype=np.int8)
        clean = np.zeros(self.n, dtype=np.uint8)
        cnt = np.zeros(1, dtype=np.uint16)
        done = np.zeros(1, dtype=np.uint8)
        lib().ssdt_step(self._map.ctypes.data, self._subs.ctypes.data, self.envs[b:b + 1].ctypes.data, self._tag[b].ctypes.data,
                        a.ctypes.data, C.byref(s) if s is not None else None, self.seed, self.gid0 + b, self.tag_timeout,
                        int(self.random_spawn_point), self.spawn_rotation,
                        reward.ctypes.data, clean.ctypes.data, cnt.ctypes.data, done.ctypes.data)
        return reward, clean, int(cnt[0]), bool(done[0])

    def obs_one(self, b=0):
        out = np.zeros((self.n, 3, self.N, self.N), dtype=np.uint8)
        lib().ssdt_render_obs(self._map.ctypes.data, self.envs[b:b + 1].ctypes.data, self._tag[b].ctypes.data, out.ctypes.data)
        return out

    def state_one(self, b=0):
        out = np.zeros((3, self.H, self.W), dtype=np.uint8)
        lib().ssdt_render_state(self._map.ctypes.data, self.envs[b:b + 1].ctypes.data, self._tag[b].ctypes.data, out.ctypes.data)
        return out

    def step(self, actions, want_obs=True, threads=1, out=None):
        a = np.ascontiguousarray(actions, dtype=np.uint8).reshape(self.B, self.n)
        if out is None:
            out = dict(reward=np.zeros((self.B, self.n), np.int8), clean=np.zeros((self.B, self.n), np.uint8),
                       apple_cnt=np.zeros(self.B, np.uint16), done=np.zeros(self.B, np.uint8),
                       obs=np.zeros((self.B, self.n, 3, self.N, self.N), np.uint8) if want_obs else None)
        lib().ssdt_batch_step(self._map.ctypes.data, self._subs.ctypes.data, self.envs.ctypes.data, self._tag.ctypes.data,
                              self.B, a.ctypes.data, self.seed, self.gid0, self.tag_timeout, int(self.random_spawn_point),
                              self.spawn_rotation, out["reward"].ctypes.data, out["clean"].ctypes.data,
                              out["apple_cnt"].ctypes.data, out["done"].ctypes.data,
                              None if not want_obs else out["obs"].ctypes.data, threads)
        return out
