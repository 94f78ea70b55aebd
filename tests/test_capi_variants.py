"""CPU suite: the per-env variant surface -- the ssd_variant layout against the header, and mapspec.compile_variant (its keys,
its errors, and LUTs equal to those compile_map derives from the same parameters)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_variant_struct_layout_matches_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    cls = _capi.SsdVariant
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ssd_b200.h"', 'int main(void) {',
             'printf("size %zu\\n", sizeof(ssd_variant));', 'printf("max %d\\n", SSD_MAX_VARIANTS);']
    lines += [f'printf("{f} %zu\\n", offsetof(ssd_variant, {f}));' for f, _ in cls._fields_]
    lines += ["return 0; }"]
    src = tmp_path / "variant.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "variant"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["size"]) == C.sizeof(cls)
    assert int(out["max"]) == _capi.SSD_MAX_VARIANTS == 256
    for f, _ in cls._fields_:
        assert int(out[f]) == getattr(cls, f).offset, f


def _base(name, mp="default5", n=5, view=7, **kw):
    from homophily_marl_b200 import mapspec
    return mapspec.compile_map(name, mp, n, view, 100, **kw)


def test_empty_overrides_are_the_base_config():
    from homophily_marl_b200 import mapspec
    for name, mp in (("cleanup", "default3"), ("cleanup", "default10"), ("harvest", "default10")):
        b = _base(name, mp, n=3, obs_color="full", fire_cost=2, hit_penalty=1, tag_timeout=4)
        v = mapspec.compile_variant(b, {})
        assert v.rows == b.rows and v.params == b.params and v.obs_color == "full"
        assert (v.fire_cost, v.hit_penalty, v.tag_timeout, v.beam_len) == (2, 1, 4, 5)
        for k in ("base_grid", "wall", "apple_pts", "waste_pts", "spawn_pts", "thr_apple", "thr_waste", "thr_harvest", "lut"):
            assert np.array_equal(getattr(v, k), getattr(b, k)), k


def test_variant_luts_equal_compile_map_with_the_same_parameters():
    from homophily_marl_b200 import mapspec
    b = _base("cleanup")
    ov = dict(threshold_depletion=0.7, threshold_restoration=0.2, waste_spawn_prob=0.4, apple_respawn_prob=0.15)
    v = mapspec.compile_variant(b, ov)
    p = mapspec.EnvParams(mapspec.KIND_CLEANUP, "cleanup_n5", **ov)
    ref = mapspec.compile_map("cleanup", "default5", 5, 7, 100, params=p)
    assert np.array_equal(v.thr_apple, ref.thr_apple) and np.array_equal(v.thr_waste, ref.thr_waste)
    assert not np.array_equal(v.thr_apple, b.thr_apple)
    h = _base("harvest", view=15)
    v = mapspec.compile_variant(h, {"spawn_prob": [0, 0.05, 0.08, 0.1], "fire_cost": 0, "tag_timeout": 9})
    ref = mapspec.compile_map("harvest", "default10", 5, 15, 100, fire_cost=0, tag_timeout=9)
    assert np.array_equal(v.thr_harvest, ref.thr_harvest) and (v.fire_cost, v.tag_timeout) == (0, 9)


def test_edited_layout_recompiles_points_and_luts():
    from homophily_marl_b200 import mapspec
    b = _base("cleanup", "default3", n=3)
    flat = "".join(b.rows).replace("H", "R", 2)
    rows = [flat[r * b.W:(r + 1) * b.W] for r in range(b.H)]
    rows[1] = "@" + rows[1][1:-2] + "@@"
    v = mapspec.compile_variant(b, {"rows": rows})
    assert len(v.waste_pts) == len(b.waste_pts) - 2 == len(v.thr_apple) - 1
    assert v.base_grid[1 * b.W + b.W - 2] == mapspec.WALL


def test_bad_overrides_raise_value_error():
    from homophily_marl_b200 import mapspec
    c, h = _base("cleanup"), _base("harvest", view=15)
    for base, ov, msg in ((c, {"spawn_prob": [0, 0, 0, 0]}, "does not apply"),
                          (h, {"waste_spawn_prob": 0.5}, "does not apply"),
                          (h, {"threshold_depletion": 0.5}, "does not apply"),
                          (c, {"view": 3}, "unknown variant key"),
                          (c, {"episode_limit": 3}, "unknown variant key"),
                          (c, {"rows": c.rows[:-1]}, "rows"),
                          (c, {"rows": [r + "@" for r in c.rows]}, "rows"),
                          (h, {"spawn_prob": [0.1, 0.2]}, "4 probabilities"),
                          (c, {"tag_timeout": 256}, "tag_timeout")):
        with pytest.raises(ValueError, match=msg):
            mapspec.compile_variant(base, ov)
