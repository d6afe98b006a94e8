"""Run the reference's OWN pytest files against this package (host engine), in place and unmodified.

`bytewax` and its submodules are aliased to `bytewax_b200` in `sys.modules`; the reference's `conftest.py`
(which imports the recovery / tracing modules that are out of scope) is cut off and its two fixtures
(`entry_point`, `now`) are provided here.  Needs a reference checkout in $BYTEWAX_SRC.

    BYTEWAX_SRC=<checkout> python tools/ref_pytests.py [pytest args / paths under $BYTEWAX_SRC/pytests]
"""
import importlib
import os
import sys
from datetime import datetime, timezone

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(os.environ.get("BYTEWAX_SRC", ""), "pytests")
sys.path.insert(0, ROOT)

ALIASES = ["", ".dataflow", ".operators", ".operators.windowing", ".operators.helpers", ".testing", ".inputs", ".outputs", ".errors", ".run",
           ".connectors", ".connectors.stdio", ".connectors.files", ".connectors.demo"]


def install_aliases():
    for a in ALIASES:
        sys.modules["bytewax" + a] = importlib.import_module("bytewax_b200" + a)


class Fixtures:
    @pytest.fixture(params=["run_main", "cluster_main-1thread", "cluster_main-2thread"])
    def entry_point_name(self, request):
        return request.param

    @pytest.fixture
    def entry_point(self, entry_point_name):
        from bytewax_b200.testing import cluster_main, run_main

        if entry_point_name == "run_main":
            return run_main
        if entry_point_name == "cluster_main-1thread":
            return lambda *a, **k: cluster_main(*a, [], 0, **k)
        return lambda *a, **k: cluster_main(*a, [], 0, worker_count_per_proc=2, **k)

    @pytest.fixture
    def now(self):
        yield datetime.now(timezone.utc)

    @pytest.fixture
    def benchmark(self):
        """pytest-benchmark is not installed: run the benchmarked callable once."""
        return lambda fn, *a, **k: fn(*a, **k)


def main(argv):
    install_aliases()
    n = next((i for i, a in enumerate(argv) if a.startswith("-")), len(argv))  # leading paths, then pytest options verbatim
    paths, opts = argv[:n] or [os.path.join(REF, "operators")], argv[n:]
    paths = [p if os.path.isabs(p) else os.path.join(REF, p) for p in paths]
    return pytest.main(paths + opts + ["-p", "no:cacheprovider", f"--confcutdir={REF}/operators", f"--rootdir={REF}",
                                       "-c", os.devnull, "-q"], plugins=[Fixtures()])


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
