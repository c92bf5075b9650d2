"""Drive the REFERENCE's own test files (tests/test_state.py, test_environment.py,
test_user_scenarios.py, test_dataloader.py -- read where they lie, never copied) against an
implementation of `explainrl.environment`:

    python tests/reference_suite_runner.py --impl adapter     # GameState / TilerSliderEnv / Factory of tiler_slider_b200
    python tests/reference_suite_runner.py --impl reference   # the reference's own classes (plumbing check)

A package `explainrl.environment` is assembled in sys.modules whose `state` and `environment`
submodules expose the chosen classes, while `display` (TextRender, which only reads attributes
of the env it is given: display.py:47-79), `dataloader` and `config` are the reference's own
files imported through the package path.  pygame / matplotlib are absent here and get empty stub
modules, as in tests/golden/make_golden.py.  The reference's suite fails 3 of its 87 tests on its
own code (SURVEY section 4: GameState.render does not exist, and a board that starts solved is
un-solved by its first move); the expected outcome for a faithful drop-in is the same 84 / 3.
Prints `passed=<n> failed=<n> failed_ids=[...]` and exits 0.
"""
import argparse
import importlib
import importlib.util
import os
import sys
import tempfile
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def install(impl: str, ref: str) -> None:
    for name in ("pygame", "matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    pkg_dir = os.path.join(ref, "explainrl")
    top = types.ModuleType("explainrl")
    top.__path__ = [pkg_dir]
    env_pkg = types.ModuleType("explainrl.environment")
    env_pkg.__path__ = [os.path.join(pkg_dir, "environment")]
    env_pkg.__package__ = "explainrl.environment"
    sys.modules["explainrl"], sys.modules["explainrl.environment"] = top, env_pkg
    top.environment = env_pkg
    if impl == "adapter":
        sys.path.insert(0, ROOT)
        import tiler_slider_b200 as ts
        st = types.ModuleType("explainrl.environment.state")
        st.GameState = ts.GameState
        en = types.ModuleType("explainrl.environment.environment")
        en.TilerSliderEnv, en.TilerSliderEnvFactory, en.GameState = ts.TilerSliderEnv, ts.TilerSliderEnvFactory, ts.GameState
        sys.modules["explainrl.environment.state"], sys.modules["explainrl.environment.environment"] = st, en
    else:
        st = importlib.import_module("explainrl.environment.state")
        en = importlib.import_module("explainrl.environment.environment")
    env_pkg.state, env_pkg.environment = st, en
    dl = importlib.import_module("explainrl.environment.dataloader")
    dp = importlib.import_module("explainrl.environment.display")
    env_pkg.GameState, env_pkg.TilerSliderEnv, env_pkg.TilerSliderEnvFactory = st.GameState, en.TilerSliderEnv, en.TilerSliderEnvFactory
    env_pkg.ImageLoader, env_pkg.TextRender, env_pkg.PygameRender = dl.ImageLoader, dp.TextRender, dp.PygameRender


class Tally:
    def __init__(self):
        self.passed, self.failed = 0, []

    def pytest_runtest_logreport(self, report):
        if report.when == "call":
            if report.passed:
                self.passed += 1
            elif report.failed:
                self.failed.append(report.nodeid.split("::", 1)[1])
        elif report.failed:
            self.failed.append(report.nodeid.split("::", 1)[1] + f" [{report.when}]")


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--impl", choices=["adapter", "reference"], default="adapter")
    ap.add_argument("--reference", default=os.environ.get("TS_REFERENCE"), required=not os.environ.get("TS_REFERENCE"),
                    help="checkout of the reference (default: $TS_REFERENCE)")
    args = ap.parse_args()
    install(args.impl, args.reference)
    import pytest
    tally = Tally()
    with tempfile.TemporaryDirectory() as tmp:      # the reference checkout is read-only: no cache, no rootdir files there
        pytest.main([os.path.join(args.reference, "tests"), "-q", "-p", "no:cacheprovider", "--rootdir", tmp, "-c", os.devnull,
                     "--disable-warnings", "-x" if False else "--tb=line"], plugins=[tally])
    print(f"passed={tally.passed} failed={len(tally.failed)} failed_ids={sorted(tally.failed)}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
