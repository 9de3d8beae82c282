"""The drop-in claim of INTEGRATION.md, executed: a copy of the reference's ``nodes/`` tree and of its own test file
(tests/test_v5_texture_ela.py of the reference, byte for byte) with ONE file replaced — nodes/V_nodes/v5_texture_ela.py by this
repo's module — and the reference's tests run against it, unmodified, by tests/dropin_runner.py in a subprocess.

The reference is not part of this repository: point V5ELA_REFERENCE_ROOT at a checkout of it to run these tests; without one they
skip. tests/test_node.py restates the same three tests against stored artefacts of the reference (tests/golden/node_golden.json),
which need no checkout. The two tests of
the reference's file that reach the analysis need the GPU (there is no CPU implementation behind the node); ``test_v5_no_faces`` and
the failure-path test run anywhere."""
import filecmp
import os
import shutil
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("V5ELA_REFERENCE_ROOT", "")
OURS = os.path.join(ROOT, "fake-video-detection-engine_b200", "nodes", "V_nodes", "v5_texture_ela.py")

pytestmark = pytest.mark.skipif(not (REF and os.path.exists(os.path.join(REF, "tests", "test_v5_texture_ela.py"))),
                                reason="needs a checkout of the reference project: set V5ELA_REFERENCE_ROOT")


@pytest.fixture
def dropin_tree(tmp_path):
    tree = tmp_path / "checkout"
    shutil.copytree(os.path.join(REF, "nodes"), tree / "nodes", ignore=shutil.ignore_patterns("__pycache__"))
    os.makedirs(tree / "tests")
    shutil.copy(os.path.join(REF, "tests", "test_v5_texture_ela.py"), tree / "tests" / "test_v5_texture_ela.py")
    shutil.copy(OURS, tree / "nodes" / "V_nodes" / "v5_texture_ela.py")           # INTEGRATION.md §1, step 3
    # nothing but the node module differs from the reference
    cmp = filecmp.dircmp(os.path.join(REF, "nodes"), tree / "nodes", ignore=["__pycache__"])
    assert cmp.diff_files == [] and cmp.left_only == [] and cmp.right_only == []
    sub = filecmp.dircmp(os.path.join(REF, "nodes", "V_nodes"), tree / "nodes" / "V_nodes", ignore=["__pycache__"])
    assert sub.diff_files == ["v5_texture_ela.py"] and sub.left_only == [] and sub.right_only == []
    assert filecmp.cmp(os.path.join(REF, "tests", "test_v5_texture_ela.py"), tree / "tests" / "test_v5_texture_ela.py", shallow=False)
    return str(tree)


def run_reference_tests(tree, *names):
    env = {k: v for k, v in os.environ.items() if k != "OPENAI_API_KEY"}
    res = subprocess.run([sys.executable, os.path.join(HERE, "dropin_runner.py"), tree, *names], capture_output=True, text=True,
                         env=env, timeout=600)
    return res.returncode, res.stdout + res.stderr


def test_reference_tests_that_need_no_device(dropin_tree):
    rc, out = run_reference_tests(dropin_tree, "TestV5TextureELA.test_v5_no_faces", "TestV5TextureELA.test_v5_openai_failure")
    assert rc == 0, out
    assert "dropin: ran 2 failures 0 errors 0" in out


@pytest.mark.gpu
def test_reference_test_file_unmodified_against_the_replaced_module(dropin_tree):
    """The reference's tests/test_v5_texture_ela.py:48-89 — all three tests, as the reference wrote them."""
    rc, out = run_reference_tests(dropin_tree)
    assert rc == 0, out
    assert "dropin: ran 3 failures 0 errors 0" in out
    assert "libv5ela" not in out or "Error analyzing face" not in out
