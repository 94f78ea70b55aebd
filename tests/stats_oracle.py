"""TEST INFRASTRUCTURE ONLY -- ``TagOracleBatch`` with the per-agent episode counters: a ctypes wrapper around
``tests/stats_oracle.c``.

``StatsOracleBatch`` steps exactly as ``TagOracleBatch`` (so with ``tag_timeout`` 0 as ``OracleBatch``) and keeps the seven counters
of DESIGN.md §3 item 16 in ``stats`` ([B, 7, n] u32, field-major like the device buffer).  Every reset zeroes the counters of the
envs it resets.  ``social_metrics`` restates the four metrics in NumPy fp64.
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
from tag_oracle import TagOracleBatch

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.join(os.path.dirname(HERE), "oracle")
N_STATS = 7
APPLES, APPLE_T, FIRES, HITS_DEALT, HITS_TAKEN, OUT_STEPS, CLEANED = range(N_STATS)
_lib = None


def build() -> str:
    srcs = [os.path.join(HERE, "stats_oracle.c"), os.path.join(HERE, "tag_oracle.c"), os.path.join(ORACLE_DIR, "ssd_oracle.c"),
            os.path.join(ORACLE_DIR, "ssd_oracle.h")]
    h = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
    out = os.path.join(tempfile.gettempdir(), f"ssd_oracle_{os.getuid()}", f"libssd_stats_oracle_{h}.so")
    if os.path.exists(out):
        return out
    os.makedirs(os.path.dirname(out), exist_ok=True)
    tmp = f"{out}.{os.getpid()}.tmp"
    base = ["-O2", "-ffp-contract=off", "-fPIC", "-std=c11", "-shared", "-I", ORACLE_DIR, "-I", HERE, "-o", tmp, srcs[0], "-lm"]
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
    raise RuntimeError("could not build the counter reference: " + " | ".join(errors))


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        P, I = C.c_void_p, C.c_int
        L.ssds_step.argtypes = [P, P, P, P, P, P, P, C.c_uint64, C.c_uint32, I, I, I, P, P, P, P]
        L.ssds_batch_step.argtypes = [P, P, P, P, P, I, P, C.c_uint64, C.c_uint32, I, I, I, P, P, P, P, P, I]
        _lib = L
    return _lib


def social_metrics(ep_ret, stats, t):
    """efficiency, equality, sustainability and peace (DESIGN.md §3 item 16) of [B, n] returns and [B, 7, n] counters after
    ``t`` steps (a scalar or [B]), in NumPy fp64."""
    r = np.asarray(ep_ret, np.float64)
    s = np.asarray(stats, np.float64)
    n = r.shape[1]
    t = np.maximum(np.broadcast_to(np.asarray(t, np.float64), r.shape[:1]), 1.0)     # t = 0: efficiency 0, peace n
    total = r.sum(1)
    denom = 2 * n * np.abs(r).sum(1)
    pair = np.abs(r[:, None, :] - r[:, :, None]).sum((1, 2))
    equality = np.where(total != 0, 1 - pair / np.where(denom == 0, 1.0, denom), 1.0)     # the runners' equality_metric
    apples, apple_t = s[:, APPLES], s[:, APPLE_T]
    ate = apples > 0
    per = np.where(ate, apple_t / np.where(ate, apples, 1.0), 0.0)
    n_ate = ate.sum(1)
    sustainability = np.where(n_ate > 0, per.sum(1) / np.maximum(n_ate, 1), 0.0)
    return dict(efficiency=total / t, equality=equality, sustainability=sustainability,
                peace=n - s[:, OUT_STEPS].sum(1) / t)


class StatsOracleBatch(TagOracleBatch):
    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self._stats = np.zeros((self.B, N_STATS, O.MAX_AGENTS), dtype=np.uint32)

    @property
    def stats(self):     # [B, 7, n]
        return self._stats[:, :, :self.n]

    def reset_one(self, b=0, draws=None):
        super().reset_one(b, draws)
        self._stats[b] = 0

    def reset(self, threads=1):
        super().reset(threads)
        self._stats[:] = 0

    def step_one(self, actions, b=0, draws=None):
        s, keep = self._draws(draws)
        a = np.ascontiguousarray(actions, dtype=np.uint8)
        reward = np.zeros(self.n, dtype=np.int8)
        clean = np.zeros(self.n, dtype=np.uint8)
        cnt = np.zeros(1, dtype=np.uint16)
        done = np.zeros(1, dtype=np.uint8)
        lib().ssds_step(self._map.ctypes.data, self._subs.ctypes.data, self.envs[b:b + 1].ctypes.data, self._tag[b].ctypes.data,
                        self._stats[b].ctypes.data, a.ctypes.data, C.byref(s) if s is not None else None, self.seed, self.gid0 + b,
                        self.tag_timeout, int(self.random_spawn_point), self.spawn_rotation,
                        reward.ctypes.data, clean.ctypes.data, cnt.ctypes.data, done.ctypes.data)
        return reward, clean, int(cnt[0]), bool(done[0])

    def step(self, actions, want_obs=True, threads=1, out=None):
        a = np.ascontiguousarray(actions, dtype=np.uint8).reshape(self.B, self.n)
        if out is None:
            out = dict(reward=np.zeros((self.B, self.n), np.int8), clean=np.zeros((self.B, self.n), np.uint8),
                       apple_cnt=np.zeros(self.B, np.uint16), done=np.zeros(self.B, np.uint8),
                       obs=np.zeros((self.B, self.n, 3, self.N, self.N), np.uint8) if want_obs else None)
        lib().ssds_batch_step(self._map.ctypes.data, self._subs.ctypes.data, self.envs.ctypes.data, self._tag.ctypes.data,
                              self._stats.ctypes.data, self.B, a.ctypes.data, self.seed, self.gid0, self.tag_timeout,
                              int(self.random_spawn_point), self.spawn_rotation, out["reward"].ctypes.data,
                              out["clean"].ctypes.data, out["apple_cnt"].ctypes.data, out["done"].ctypes.data,
                              None if not want_obs else out["obs"].ctypes.data, threads)
        return out

    def social_metrics(self, t=None):
        return social_metrics(self.ep_ret, self.stats, self.envs["t"] if t is None else t)
