"""Install the original ShallowSpeed project into ``oracle/_ref/`` so that ``bench.py --impl reference`` (via
``baseline/run_reference.py``) can run it unmodified next to this one.

The original is pure Python (one package, ``shallowspeed``, with NumPy / pandas as its only dependencies), so
installing it means copying that package's modules; ``oracle/_ref/`` is git-ignored.  ``build()`` calls
``install()``: the source is ``$SSB_REFERENCE_SRC`` or, by default, a checkout mounted read-only at
``DEFAULT_SOURCE``.  Without a source an existing install is kept and nothing fails: only the reference arm of
the benchmark and its test need it.

    python oracle/install_reference.py [SOURCE]
"""
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
TARGET = os.path.join(HERE, "_ref")
DEFAULT_SOURCE = "/root/reference"
PACKAGE = "shallowspeed"


def installed() -> bool:
    return os.path.exists(os.path.join(TARGET, PACKAGE, "pipe.py"))


def install(source=None) -> bool:
    """Copy ``<source>/shallowspeed/*.py`` to ``oracle/_ref/shallowspeed/``; True when an install is present after."""
    source = source or os.environ.get("SSB_REFERENCE_SRC") or DEFAULT_SOURCE
    src_pkg = os.path.join(source, PACKAGE)
    if not os.path.isfile(os.path.join(src_pkg, "pipe.py")):
        return installed()
    dst_pkg = os.path.join(TARGET, PACKAGE)
    shutil.rmtree(TARGET, ignore_errors=True)
    os.makedirs(dst_pkg)
    for name in sorted(os.listdir(src_pkg)):
        if name.endswith(".py"):
            shutil.copyfile(os.path.join(src_pkg, name), os.path.join(dst_pkg, name))   # contents only: stays writable
    return installed()


if __name__ == "__main__":
    ok = install(sys.argv[1] if len(sys.argv) > 1 else None)
    print("oracle/_ref:", "installed" if ok else "not installed (original project not found)")
    sys.exit(0 if ok else 1)
