"""oracle/_ref/: the reference (dpwe/audfprint, pure Python) compiled to sourceless bytecode,
with the MP3 files its own `make test` uses.  Some tests run the reference's OWN code - its
command line on the mirror classes (tests/test_reference_cli_cpu.py), its decoding and command
line on the bundled audio (tests/test_oracle_bundled.py) - and read it from here, so they run
wherever the built tree goes, with or without the checkout beside it.

__graft_entry__.build() calls build(): it compiles the checkout named by $AFP_REFERENCE, else
the one at DEFAULT_CHECKOUT, and leaves oracle/_ref/ as it is when neither exists.
oracle/_ref/ is a build product and stays out of git; no reference source is stored in it.
"""
from __future__ import annotations

import glob
import os
import py_compile
import shutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "oracle", "_ref")
DEFAULT_CHECKOUT = "/root/reference"        # where the reference checkout is conventionally mounted


def checkout():
    """The reference checkout to compile, or None."""
    d = os.environ.get("AFP_REFERENCE") or DEFAULT_CHECKOUT
    return d if os.path.isfile(os.path.join(d, "audfprint.py")) else None


def build():
    """(Re)write oracle/_ref/ from the checkout: <module>.pyc for every top-level module, which
    Python imports without a source file, and tests/data/ copied as it is."""
    src = checkout()
    if src is None:
        return None
    tmp = OUT + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    os.makedirs(tmp)
    for py in sorted(glob.glob(os.path.join(src, "*.py"))):
        name = os.path.basename(py)
        if name != "__init__.py":
            py_compile.compile(py, cfile=os.path.join(tmp, name + "c"), doraise=True)
    shutil.copytree(os.path.join(src, "tests", "data"), os.path.join(tmp, "tests", "data"))
    for dirpath, dirnames, filenames in os.walk(tmp):          # the checkout may be read-only
        for n in dirnames + filenames:
            os.chmod(os.path.join(dirpath, n), 0o755 if n in dirnames else 0o644)
    shutil.rmtree(OUT, ignore_errors=True)
    os.replace(tmp, OUT)
    return OUT


def reference_dir():
    """Where the tests find the reference's code: $AFP_REFERENCE if it names a checkout, else
    oracle/_ref/ if build() made it, else None."""
    d = os.environ.get("AFP_REFERENCE")
    if d and os.path.isfile(os.path.join(d, "audfprint.py")):
        return d
    return OUT if os.path.isfile(os.path.join(OUT, "audfprint.pyc")) else None
