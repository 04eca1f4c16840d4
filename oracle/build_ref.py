"""Byte-compile the reference PyDESeq2 package into ``oracle/_ref/pydeseq2`` (sourceless ``.pyc`` files, not tracked by git).

The drop-in tests (tests/test_reference_dropin.py) run the reference's own orchestrator with the B200 backend plugged in; the
shim ``oracle/refshim/pydeseq2`` imports the package from this directory, so the tests run wherever it was built, including
machines without the reference checkout.  The checkout is found at ``$PDQ_REFERENCE`` (default ``/root/reference``); without
it nothing is compiled and an existing ``_ref`` is left as it is.
"""
from __future__ import annotations

import glob
import os
import py_compile

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref", "pydeseq2")


def build() -> str | None:
    src = os.path.join(os.environ.get("PDQ_REFERENCE", "/root/reference"), "pydeseq2")
    files = sorted(glob.glob(os.path.join(src, "*.py")))
    if not files:
        return None
    os.makedirs(OUT, exist_ok=True)
    for f in files:
        name = os.path.splitext(os.path.basename(f))[0]
        py_compile.compile(f, cfile=os.path.join(OUT, name + ".pyc"), doraise=True,
                           invalidation_mode=py_compile.PycInvalidationMode.UNCHECKED_HASH)
    return OUT


if __name__ == "__main__":
    print(build())
