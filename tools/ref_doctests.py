"""Run the `{testcode}` / `{testoutput}` examples of the reference's operator docstrings against this package.

The reference documents every operator with a runnable example and its expected stdout (Sphinx doctest blocks in
pysrc/bytewax/operators/__init__.py and windowing.py).  This extracts them from the reference tree in place, runs each
example with `bytewax` aliased to `bytewax_b200`, and compares stdout.  Needs a reference checkout in $BYTEWAX_SRC.

    BYTEWAX_SRC=<checkout> python tools/ref_doctests.py            # summary; exit code 1 if any example differs
"""
import ast
import contextlib
import io
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_ROOT = os.environ.get("BYTEWAX_SRC", "")
REF = os.path.join(REF_ROOT, "pysrc", "bytewax")
sys.path.insert(0, os.path.join(ROOT, "compat"))
sys.path.insert(0, ROOT)

BLOCK = re.compile(r"```\{(testcode|testoutput)\}\n(.*?)```", re.S)


def examples(path):
    """(qualified name, code, expected stdout) for every docstring that has at least one testoutput block."""
    tree = ast.parse(open(path).read())
    for node in ast.walk(tree):
        if not isinstance(node, (ast.FunctionDef, ast.ClassDef, ast.Module)):
            continue
        doc = ast.get_docstring(node, clean=True)
        if not doc or "{testoutput}" not in doc:
            continue
        code, want = [], []
        for kind, body in BLOCK.findall(doc):
            body = "\n".join(ln for ln in body.split("\n") if not ln.strip().startswith(":hide:"))
            (code if kind == "testcode" else want).append(body)
        yield getattr(node, "name", "<module>"), "\n".join(code), "\n".join(want)


def md_examples(path):
    """A guide page is one running session: code blocks accumulate; each testoutput block checks the stdout produced since
    the previous one."""
    text = open(path).read()
    code = []
    for kind, body in BLOCK.findall(text):
        body = "\n".join(ln for ln in body.split("\n") if not ln.strip().startswith(":hide:"))
        if kind == "testcode":
            code.append(body)
        else:
            yield "\n".join(code), body
            code = []


def run_guides(names):
    """(ok, bad) over the guide pages: every page runs in one namespace, cwd = docs/fixtures (pages read sample files)."""
    ok, bad = 0, []
    docs = os.path.join(REF_ROOT, "docs", "guide")
    cwd = os.getcwd()
    os.chdir(os.path.join(REF_ROOT, "docs", "fixtures"))  # the pages' doctests run beside their fixture files
    try:
        for rel in names:
            ns = {"__name__": "__doctest__"}
            for i, (code, want) in enumerate(md_examples(os.path.join(docs, rel))):
                buf = io.StringIO()
                try:
                    with contextlib.redirect_stdout(buf):
                        exec(compile(code, f"<{rel}#{i}>", "exec"), ns)
                    if norm(buf.getvalue()) == norm(want):
                        ok += 1
                    else:
                        bad.append((rel, i, "stdout differs", norm(buf.getvalue())[:5], norm(want)[:5]))
                except Exception as ex:  # noqa: BLE001
                    bad.append((rel, i, f"{type(ex).__name__}: {ex}"[:200], [], []))
    finally:
        os.chdir(cwd)
    return ok, bad


def norm(s):
    return [ln.rstrip() for ln in s.strip().split("\n") if ln.strip()]


def main():
    ok, bad = 0, []
    for rel in ("operators/__init__.py", "operators/windowing.py", "operators/helpers.py", "dataflow.py", "inputs.py", "testing.py"):
        path = os.path.join(REF, rel)
        if not os.path.exists(path):
            continue
        for name, code, want in examples(path):
            buf = io.StringIO()
            try:
                with contextlib.redirect_stdout(buf):
                    exec(compile(code, f"<{rel}:{name}>", "exec"), {"__name__": "__doctest__"})
                got = buf.getvalue()
                if norm(got) == norm(want):
                    ok += 1
                else:
                    bad.append((rel, name, "stdout differs", norm(got)[:6], norm(want)[:6]))
            except Exception as ex:  # noqa: BLE001
                bad.append((rel, name, f"{type(ex).__name__}: {ex}"[:200], [], []))
    print(f"{ok} docstring examples reproduce the documented output; {len(bad)} do not")
    for b in bad:
        print("  ", b)
    if "--guides" in sys.argv:
        gok, gbad = run_guides(["concepts/joins.md", "concepts/dataflow-programming.md", "getting-started/wordcount-example.md",
                                "getting-started/collecting-windowing-example.md", "getting-started/join-example.md",
                                "getting-started/simple-example.md"])
        print(f"{gok} guide-page examples reproduce the documented output; {len(gbad)} do not")
        for b in gbad:
            print("  ", b)
        bad += gbad
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
