"""Copy the unmodified reference's `core/` package (abdo-eldesokey/RAFT-NCUP, pure Python) into the git-ignored oracle/_ref/ for
bench.py's `--impl reference` and `gpu_eager_baseline` legs.  oracle/_ref/ is a build product: it is made once by build() on a
machine that has a checkout of the reference and travels with the working tree; bench.py falls back to the oracle port without it.

    python oracle/install_reference.py [REFERENCE_CHECKOUT]

The checkout is the argument, else $RNC_REFERENCE, else a directory `reference` beside this repository.
"""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "oracle", "_ref")


def reference_checkout(path=None):
    return path or os.environ.get("RNC_REFERENCE") or os.path.join(os.path.dirname(ROOT), "reference")


def install(path=None):
    """Returns oracle/_ref/core when it exists afterwards, else None (no readable reference checkout)."""
    src = os.path.join(reference_checkout(path), "core")
    dst = os.path.join(DST, "core")
    if os.path.exists(os.path.join(dst, "raft_nc_dbl.py")):
        return dst
    if not os.access(os.path.join(src, "raft_nc_dbl.py"), os.R_OK):
        return None
    shutil.rmtree(DST, ignore_errors=True)
    for d, dirs, files in os.walk(src):
        dirs[:] = [x for x in dirs if x != "__pycache__"]
        out = os.path.join(dst, os.path.relpath(d, src))
        os.makedirs(out, exist_ok=True)
        for f in files:
            if f.endswith(".py"):
                shutil.copyfile(os.path.join(d, f), os.path.join(out, f))       # contents only: the copy stays writable
    return dst


if __name__ == "__main__":
    print(install(sys.argv[1] if len(sys.argv) > 1 else None) or "no reference checkout found: nothing installed")
