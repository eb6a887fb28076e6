"""GPU: parity cases through the CHECKED build of the library (csrc/libccb200_checked.so: the same sources compiled with
-DCCB_CHECKS, i.e. device-side asserts on every data-dependent shared-memory index, on the policy bitmap that aliases the
TMA image ring and on the bulk-copy sizes).  compute-sanitizer is closed on this pool
(profiles/r2_compute_sanitizer_closed_on_this_pool.txt); a failed assert traps the kernel and fails the run."""

import os
import subprocess
import sys
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]
CHECKED = ROOT / "collectivecrossing_b200" / "csrc" / "libccb200_checked.so"


def test_parity_cases_pass_in_the_checked_build():
    if not CHECKED.exists():
        pytest.skip("checked library not built (make -C collectivecrossing_b200/csrc libccb200_checked.so)")
    env = dict(os.environ, CCB200_LIB=str(CHECKED))
    sel = ["tests/test_gpu_small_lattice.py", "tests/test_gpu_host_path.py::test_table_mode_matches_oracle",
           "tests/test_gpu_parity.py::test_device_matches_oracle_with_auto_reset", "tests/test_gpu_parity.py::test_fused_rollout_equals_repeated_steps",
           "tests/test_gpu_parity.py::test_thread_per_env_kernel_replays_golden",
           "tests/test_gpu_geometry_edges.py"]
    proc = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", *sel], cwd=ROOT, env=env,
                          capture_output=True, text=True, timeout=1500)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0, tail
    assert " passed" in tail and "failed" not in tail, tail
