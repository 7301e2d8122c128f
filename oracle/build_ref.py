"""TEST INFRASTRUCTURE -- byte-compile an unmodified CFDBench `src/` tree into the git-ignored oracle/_ref/src/.

    python oracle/build_ref.py [CFDBENCH_SRC]

The reference is a pure-Python script tree, so its build product is bytecode: every module becomes a sourceless
`<name>.pyc` at its own path (no source text is stored), which Python imports and `runpy` runs like the source.
`tests/test_gpu_runner.py` runs the reference's scripts from here and `bench.py`'s CPU baseline times its `Fno2d`.
The source tree is CFDBENCH_SRC, else DEFAULT_SRC; without either, nothing is built and those fall back or skip.
The bytecode matches the interpreter that built it, so build and run with the same Python.
"""
from __future__ import annotations

import os
import py_compile
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref", "src")
DEFAULT_SRC = "/root/reference/src"   # where an unmodified CFDBench checkout is looked for when CFDBENCH_SRC is unset


def source_dir() -> str:
    return os.environ.get("CFDBENCH_SRC") or DEFAULT_SRC


def build(src: str | None = None) -> str | None:
    """Compile `src` into DST (replacing what was there); returns DST, or None when there is no readable tree."""
    src = os.path.abspath(src or source_dir())
    if not os.path.isdir(os.path.join(src, "models", "fno")):
        return None
    tmp = DST + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    for dirpath, dirnames, filenames in os.walk(src):
        dirnames[:] = sorted(d for d in dirnames if d != "__pycache__")
        rel_dir = os.path.relpath(dirpath, src)
        for name in sorted(filenames):
            if name.endswith(".py"):
                rel = os.path.normpath(os.path.join(rel_dir, name))
                py_compile.compile(os.path.join(dirpath, name), cfile=os.path.join(tmp, rel + "c"),
                                   dfile=rel, doraise=True)
    shutil.rmtree(DST, ignore_errors=True)
    os.replace(tmp, DST)
    return DST


if __name__ == "__main__":
    out = build(sys.argv[1] if len(sys.argv) > 1 else None)
    print(out or f"no CFDBench src/ tree at {source_dir()}: nothing built")
