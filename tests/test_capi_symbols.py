"""CPU suite: the C-ABI library loads without a GPU, exports every symbol include/ssd_b200.h declares,
its struct layouts match the ctypes mirror, argument validation works before any CUDA call, and the
product path fails loudly (no CPU fallback)."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from harness import ssd_config

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HDR = os.path.join(ROOT, "include", "ssd_b200.h")


@pytest.fixture(scope="module")
def lib():
    from homophily_marl_b200 import _build, _capi
    _build.build()
    return _capi.load()


def declared_functions():
    text = open(HDR).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(ssd_[a-z0-9_]+)\s*\(", text)))


def test_every_declared_symbol_is_exported(lib):
    from homophily_marl_b200 import _capi
    names = declared_functions()
    assert len(names) >= 13
    for n in names:
        assert hasattr(lib, n), n
    assert sorted(_capi.EXPORTS) == names
    assert lib.ssd_abi_version() == 2
    assert lib.ssd_error_string(-3).decode().startswith("There are not enough spawn points")


def test_struct_layouts_match_the_header(tmp_path):
    from homophily_marl_b200 import _capi
    structs = {"ssd_config": _capi.SsdConfig, "ssd_layout": _capi.SsdLayout, "ssd_state": _capi.SsdState,
               "ssd_step_out": _capi.SsdStepOut, "ssd_draws": _capi.SsdDraws}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "ssd_b200.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for f, _ in cls._fields_:
            lines.append(f'printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));')
    lines += ["return 0; }"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
    subprocess.run([cc, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    out = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == C.sizeof(cls), cname
        for f, _ in cls._fields_:
            assert int(out[f"{cname}.{f}"]) == getattr(cls, f).offset, (cname, f)


def test_prob_to_threshold_matches_host_compiler(lib):
    from homophily_marl_b200 import mapspec
    for p in (0.0, -1.0, 1e-12, 0.005, 0.02, 0.05, 0.08, 0.1, 0.3, 0.20625, 0.11249999999999999, 0.5, 0.999999, 1.0, 2.0):
        assert lib.ssd_prob_to_threshold(p) == mapspec.prob_to_threshold(p), p
    k = np.arange(0, 2 ** 32, 2 ** 20, dtype=np.uint64)
    for p in (0.05, 0.3, 0.5):
        T = mapspec.prob_to_threshold(p)
        assert np.array_equal(k / 2.0 ** 32 < p, k < T)


def test_create_validates_before_touching_cuda(lib):
    from homophily_marl_b200 import _capi
    h = C.c_void_p()
    ok_rows = ["@@@@@", "@P B@", "@ P @", "@@@@@"]
    assert lib.ssd_create(C.byref(ssd_config(["@@@@@", "@P B ", "@ P @", "@@@@@"])), C.byref(h)) == _capi.SSD_ERR_MAP      # open border
    assert lib.ssd_create(C.byref(ssd_config(["@@@@@", "@P x@", "@ P @", "@@@@@"])), C.byref(h)) == _capi.SSD_ERR_MAP      # unknown char
    assert lib.ssd_create(C.byref(ssd_config(ok_rows, n=3)), C.byref(h)) == _capi.SSD_ERR_SPAWN                            # map_env.py:783
    assert lib.ssd_create(C.byref(ssd_config(ok_rows, n=17)), C.byref(h)) == _capi.SSD_ERR_INVALID
    assert lib.ssd_create(C.byref(ssd_config(ok_rows, kind=5)), C.byref(h)) == _capi.SSD_ERR_INVALID
    assert lib.ssd_create(C.byref(ssd_config(ok_rows, hit_penalty=127)), C.byref(h)) == _capi.SSD_ERR_INVALID              # int8 reward
    assert lib.ssd_create(None, C.byref(h)) == _capi.SSD_ERR_INVALID
    assert lib.ssd_step(None, None, None, None, None, None) == _capi.SSD_ERR_INVALID
    assert lib.ssd_destroy(None) == _capi.SSD_ERR_INVALID


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from homophily_marl_b200 import _capi
    from homophily_marl_b200.batch_env import SSDBatchEnv
    from homophily_marl_b200.pymarl_env import REGISTRY
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        SSDBatchEnv("cleanup", 4, 5, map="default5")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        REGISTRY["harvest"](num_agents=5, map="default10", view_size=15, quiet=True)
    lib = _capi.load()
    h = C.c_void_p()
    rc = lib.ssd_create(C.byref(ssd_config(["@@@@@", "@P B@", "@ P @", "@@@@@"])), C.byref(h))
    assert rc == _capi.SSD_ERR_CUDA and lib.ssd_last_cuda_error() != 0


def test_product_never_imports_the_oracle():
    """The oracle is test infrastructure: nothing under homophily_marl_b200/ may reference it."""
    pkg = os.path.join(ROOT, "homophily_marl_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cuh")):
                text = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in text.lower().replace("# the oracle is", ""), os.path.join(dirpath, f)
    code = "import sys; sys.path.insert(0, %r); import homophily_marl_b200, homophily_marl_b200.mapspec, homophily_marl_b200._capi; " \
           "assert not [m for m in sys.modules if m.startswith('oracle')]" % ROOT
    subprocess.run([sys.executable, "-c", code], check=True)
