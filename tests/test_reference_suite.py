"""The reference's OWN test files (tests/collectivecrossing/envs/*.py) run unmodified

* against the unmodified reference behind the stub gymnasium / ray / matplotlib modules (CPU; validates the
  harness, the stubs and the staged archive), and
* against the drop-in façade: ``sys.modules["collectivecrossing"]`` and ``baseline_policies`` are aliased to
  ``collectivecrossing_b200`` before the files are imported (GPU: every step is a kernel launch).

The files come from /root/reference when it is mounted, else from the archive oracle/stage_ref.py staged
(oracle/_ref/reference.zip, which travels to the GPU box); without either the tests skip."""

import re
import subprocess
import sys
import textwrap
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parents[1]

CONFTEST_REFERENCE = """
import sys
sys.path.insert(0, {root!r})
from oracle import refload
refload.load()   # stubs + the reference package itself on sys.path
"""

CONFTEST_FACADE = """
import importlib, sys
sys.path.insert(0, {root!r})
from oracle import refload
refload._install_stubs()   # gymnasium / ray / matplotlib stand-ins only; the package under test is ours
import collectivecrossing_b200 as pkg
sys.modules["collectivecrossing"] = pkg
for sub in ("collectivecrossing", "configs", "reward_configs", "terminated_configs", "truncated_configs", "observation_configs",
            "rewards", "terminateds", "truncateds", "observations", "types", "actions", "utils", "utils.geometry", "utils.pydantic"):
    sys.modules["collectivecrossing." + sub] = importlib.import_module("collectivecrossing_b200." + sub)
bp = importlib.import_module("collectivecrossing_b200.baseline_policies")
sys.modules["baseline_policies"] = bp
for sub in ("greedy_policy", "waiting_policy"):
    sys.modules["baseline_policies." + sub] = importlib.import_module("collectivecrossing_b200.baseline_policies." + sub)
"""


def run_suite(tmp_path: Path, conftest: str) -> tuple[int, int, str]:
    from oracle import refload

    if not refload.available():
        pytest.skip("reference neither mounted nor staged (oracle/_ref/reference.zip)")
    root = refload.extract(tmp_path / "ref", prefixes=("tests/",))
    (root / "tests" / "conftest.py").write_text(textwrap.dedent(conftest).format(root=str(ROOT)))
    (root / "pytest.ini").write_text("[pytest]\ntestpaths = tests\n")
    # test_rendering draws a 1200x800 matplotlib figure: rendering is out of scope (SURVEY.md §2) and matplotlib is not installed
    proc = subprocess.run([sys.executable, "-m", "pytest", "tests/collectivecrossing/envs", "-q", "-p", "no:cacheprovider", "--tb=short",
                           "-c", "pytest.ini", "--rootdir", str(root),
                           "--deselect", "tests/collectivecrossing/envs/test_collective_crossing.py::test_rendering"],
                          cwd=root, capture_output=True, text=True, timeout=1500)
    out = proc.stdout + proc.stderr
    m_pass, m_fail = re.search(r"(\d+) passed", out), re.search(r"(\d+) (?:failed|error)", out)
    return (int(m_pass.group(1)) if m_pass else 0), (int(m_fail.group(1)) if m_fail else 0), out


def test_reference_suite_passes_on_the_reference_behind_the_stubs(tmp_path):
    passed, failed, out = run_suite(tmp_path, CONFTEST_REFERENCE)
    assert failed == 0 and passed >= 60, out[-4000:]


@pytest.mark.gpu
def test_reference_suite_passes_on_the_facade(tmp_path):
    passed, failed, out = run_suite(tmp_path, CONFTEST_FACADE)
    assert failed == 0 and passed >= 60, out[-6000:]
