"""GPU suite: the checked build (libssd_b200_check.so, -DSSD_BOUNDS_CHECK) sees no shared-memory index violation.

The checked library tests every data-dependent shared-memory index against its tile and counts the violations.  It is a
different library, chosen when ``_capi`` loads, so one pytest subprocess with SSD_B200_CHECKED=1 runs the GPU tests in NODES on
it; the session fixture ``_checked_build_reports_no_violation`` in conftest.py fails that run unless ``ssd_debug_oob_count()``
is 0 at its end.  A node id that no longer exists makes the run fail, so the list cannot go stale unnoticed."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# specialised and runtime geometry, tagging, both colour schemes, all four (obs, state) formats, auto-reset and variants
NODES = [
    # index4 observations: shipped maps with and without tagging, and the custom maps of the runtime geometry
    "tests/test_gpu_obs_index.py::test_every_config_matches_reference[cleanup10_full-full-0]",
    "tests/test_gpu_obs_index.py::test_every_config_matches_reference[cleanup10_full-full-3]",
    "tests/test_gpu_obs_index.py::test_every_config_matches_reference[harvest5-simplified-0]",
    "tests/test_gpu_obs_index.py::test_every_config_matches_reference[harvest5-simplified-3]",
    "tests/test_gpu_obs_index.py::test_every_config_matches_reference[harvest10_full-full-0]",
    "tests/test_gpu_obs_index.py::test_every_config_matches_reference[harvest10_full-full-3]",
    "tests/test_gpu_obs_index.py::test_runtime_geometry_custom_maps",
    # index4 state images
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[cleanup3-simplified-0]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[cleanup3-simplified-3]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[cleanup10_full-full-0]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[cleanup10_full-full-3]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[harvest5-simplified-0]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[harvest5-simplified-3]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[harvest10_full-full-0]",
    "tests/test_gpu_state_index.py::test_every_config_matches_reference[harvest10_full-full-3]",
    "tests/test_gpu_state_index.py::test_runtime_geometry_custom_maps",
    # tagging-out timers
    "tests/test_gpu_tagging.py::test_every_config_matches_oracle_with_tagging[cleanup10_full]",
    "tests/test_gpu_tagging.py::test_every_config_matches_oracle_with_tagging[harvest5]",
    "tests/test_gpu_tagging.py::test_every_config_matches_oracle_with_tagging[harvest10_full]",
    # auto-reset in the step launch, and on the runtime geometry (SSD_B200_GENERIC=1 and a custom map)
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[cleanup5-simplified-0]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[cleanup5-simplified-3]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[cleanup5-full-0]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[cleanup5-full-3]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest5-simplified-0]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest5-simplified-3]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest5-full-0]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest5-full-3]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest10_full-simplified-0]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest10_full-simplified-3]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest10_full-full-0]",
    "tests/test_gpu_autoreset.py::test_fused_equals_the_three_launch_sequence[harvest10_full-full-3]",
    "tests/test_gpu_autoreset.py::test_runtime_geometry_matches_the_oracle",
    # per-env variants, also on the runtime geometry
    "tests/test_gpu_variants.py::test_mixed_batch_equals_single_config_twins[harvest5-autoreset]",
    "tests/test_gpu_variants.py::test_mixed_batch_equals_single_config_twins[cleanup10-step]",
    "tests/test_gpu_variants.py::test_runtime_geometry_kernels",
    # every kernel mode on both envs and both geometries, injected draws
    "tests/test_gpu_generic_geometry.py::test_all_paths_workload",
]


def test_checked_build_sees_no_shared_memory_violation():
    from homophily_marl_b200 import _build
    _build.build_checked()
    r = subprocess.run([sys.executable, "-m", "pytest", "-p", "no:cacheprovider", "-q", "-rA", "-m", "gpu"] + NODES, cwd=ROOT,
                       env={**os.environ, "SSD_B200_CHECKED": "1"}, capture_output=True, text=True, timeout=3600)
    print(r.stdout[-20000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    passed = [line.split()[1] for line in r.stdout.splitlines() if line.startswith("PASSED ")]
    for node in NODES:
        assert any(p == node or p.startswith(node + "[") for p in passed), node
