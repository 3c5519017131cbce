"""Run the reference's OWN test files, unmodified, against this package on the GPU.

The files are staged by __graft_entry__.build() (oracle/build_ref.stage_tests()) from the reference checkout
($TSB200_REFERENCE, else `reference` beside this repository) into oracle/_ref/ref_tests/ (git-ignored like the rest of
oracle/_ref: the reference's sources never enter this repository's history); without them the test skips.
`torch_sparse` resolves to tests/ref_shim/torch_sparse (:= pytorch_sparse_b200), `torch_scatter` to the pure-torch
stand-in the tests use to build expected values. Expected outcome of every test id: tests/golden/ref_suite_outcomes.json (all 109 test ids pass since SparseStorage / SparseTensor are TorchScript classes;
tests/ref_suite_xfail.json would hold reasons for expected failures — it is empty)."""
import json
import os
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
STAGED = ROOT / "oracle" / "_ref" / "ref_tests"
EXPECTED = ROOT / "tests" / "golden" / "ref_suite_outcomes.json"
FILES = ["test_matmul.py", "test_spmm.py", "test_spspmm.py", "test_coalesce.py", "test_storage.py",
         "test_transpose.py", "test_add.py", "test_mul.py", "test_tensor.py", "test_overload.py"]


@pytest.mark.gpu
def test_reference_suite_runs_green(tmp_path):
    files = [STAGED / f for f in FILES if (STAGED / f).exists()]
    if not files:
        pytest.skip("oracle/_ref/ref_tests not staged (run __graft_entry__.build() with a checkout of the reference at hand)")
    report = tmp_path / "outcomes.json"
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([str(ROOT / "tests" / "ref_shim"), str(ROOT / "oracle" / "torch_scatter_standin"),
                                         str(ROOT), env.get("PYTHONPATH", "")])
    env["TSB200_REF_REPORT"] = str(report)
    res = subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "tsb200_ref_plugin",
                          "-p", "no:cacheprovider", "--rootdir", str(STAGED), "-c", os.devnull, *map(str, files)],
                         capture_output=True, text=True, env=env, cwd=str(tmp_path), timeout=1500)
    tail = (res.stdout + res.stderr)[-6000:]
    got = json.loads(report.read_text()) if report.exists() else {}
    assert res.returncode == 0, tail
    assert got and all(v in ("passed", "xfailed", "xpassed") for v in got.values()), tail
    if EXPECTED.exists():   # nothing that is expected to pass may have stopped passing, and no test id may be missing
        want = json.loads(EXPECTED.read_text())
        worse = {k: (w, got.get(k)) for k, w in want.items()
                 if got.get(k) is None or (w == "passed" and got.get(k) not in ("passed", "xpassed"))}
        assert not worse, worse
