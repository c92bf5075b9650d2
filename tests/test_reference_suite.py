"""SURVEY 8(f) N1: the reference's own test files driven, unchanged, against the drop-in adapter.

The reference checkout is not part of this repository: both tests run only where $TS_REFERENCE
names it, the adapter run only where a CUDA device is present too.  The plumbing check needs no
GPU: the same runner with the reference's own classes behind the assembled
`explainrl.environment` package must reproduce the reference's known 84 passed / 3 failed."""
import ast
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("TS_REFERENCE", "")
KNOWN_REFERENCE_FAILURES = ["TestEdgeCases::test_already_won_initial_state", "TestRendering::test_render_basic",
                            "TestRendering::test_render_multi_color"]
needs_reference = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "tests")),
                                     reason="needs $TS_REFERENCE: a checkout of the reference with its tests/")


def _run(impl):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "reference_suite_runner.py"), "--impl", impl,
                          "--reference", REF], capture_output=True, text=True, timeout=900)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("passed=")]
    assert line, out.stdout[-3000:] + out.stderr[-3000:]
    fields = dict(kv.split("=", 1) for kv in line[-1].split(" ", 2))
    return int(fields["passed"]), int(fields["failed"]), ast.literal_eval(fields["failed_ids"])


@needs_reference
def test_runner_reproduces_the_reference_on_its_own_classes():
    passed, failed, ids = _run("reference")
    assert (passed, failed) == (84, 3) and ids == KNOWN_REFERENCE_FAILURES


@pytest.mark.gpu
@needs_reference
def test_reference_suite_against_the_cuda_adapter():
    """Same files, GameState / TilerSliderEnv / TilerSliderEnvFactory of tiler_slider_b200 behind
    them, the reference's TextRender on top: a faithful drop-in fails exactly the reference's own
    three tests (missing GameState.render x2; no 'already won' short circuit) and passes the rest."""
    passed, failed, ids = _run("adapter")
    assert ids == KNOWN_REFERENCE_FAILURES and passed == 84, (passed, failed, ids)
