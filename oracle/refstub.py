"""Import the reference's *Python half* in place.  TEST INFRASTRUCTURE ONLY.

Works only where a source checkout of the reference (bytewax v0.21.1) is given
in ``$BYTEWAX_SRC``.  Used by ``oracle/gen_golden.py`` to produce
``tests/golden/*``.

The reference's engine is Rust (``bytewax._bytewax``, src/lib.rs:24-32) and
cannot be built here (no cargo, un-vendored timely; SURVEY.md section 8c).  Its
Python operator logic imports fine once a stub ``bytewax._bytewax`` with the
13 names of ``pysrc/bytewax/_bytewax.pyi`` is registered first.
"""

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("BYTEWAX_SRC", "")
REFERENCE_PYSRC = os.path.join(REFERENCE_ROOT, "pysrc") if REFERENCE_ROOT else ""


def available() -> bool:
    return bool(REFERENCE_PYSRC) and os.path.isdir(os.path.join(REFERENCE_PYSRC, "bytewax"))


def load():
    """Return the reference's ``bytewax.operators.windowing`` module."""
    if not available():
        raise RuntimeError("reference checkout not found: set BYTEWAX_SRC to a bytewax v0.21.1 source tree")
    if "bytewax" in sys.modules and not getattr(sys.modules["bytewax"], "__file__", "").startswith(
        REFERENCE_PYSRC
    ):
        raise RuntimeError("a different `bytewax` is already imported")
    if "bytewax._bytewax" not in sys.modules:
        stub = types.ModuleType("bytewax._bytewax")

        class AbortExecution(RuntimeError):
            pass

        class InconsistentPartitionsError(ValueError):
            pass

        class MissingPartitionsError(FileNotFoundError):
            pass

        class NoPartitionsError(FileNotFoundError):
            pass

        class RecoveryConfig:
            def __init__(self, db_dir, backup_interval=None):
                self.db_dir, self.backup_interval = db_dir, backup_interval

        class TracingConfig:
            pass

        class JaegerConfig(TracingConfig):
            pass

        class OtlpTracingConfig(TracingConfig):
            pass

        def _unavailable(*_a, **_k):
            raise RuntimeError("the reference's Rust engine is not built here")

        for name, obj in dict(
            AbortExecution=AbortExecution,
            InconsistentPartitionsError=InconsistentPartitionsError,
            MissingPartitionsError=MissingPartitionsError,
            NoPartitionsError=NoPartitionsError,
            RecoveryConfig=RecoveryConfig,
            TracingConfig=TracingConfig,
            JaegerConfig=JaegerConfig,
            OtlpTracingConfig=OtlpTracingConfig,
            init_db_dir=_unavailable,
            setup_tracing=_unavailable,
            run_main=_unavailable,
            cluster_main=_unavailable,
            cli_main=_unavailable,
        ).items():
            setattr(stub, name, obj)
        sys.modules["bytewax._bytewax"] = stub
    if REFERENCE_PYSRC not in sys.path:
        sys.path.insert(0, REFERENCE_PYSRC)
    import bytewax.operators.windowing as win  # noqa: E402

    return win


def find_stateful_batch(flow):
    """Depth-first search of ``flow.substeps`` for the ``stateful_batch`` core step
    (src/worker.rs:289-293, 447-461)."""
    stack = list(flow.substeps)
    while stack:
        step = stack.pop(0)
        if type(step).__name__ == "stateful_batch":
            return step
        stack = list(getattr(step, "substeps", [])) + stack
    raise LookupError("no stateful_batch step")
