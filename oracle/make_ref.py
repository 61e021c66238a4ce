"""Populate oracle/_ref/ with a read-only copy of the reference's Python package (SURVEY.md 7 step 0, 8c).
The directory is git-ignored: the copy never enters history.  tests/test_adapter_cpu.py, tests/test_gpu_reference.py and
`bench.py --impl reference` import it through oracle/ref_shims and skip (or time the oracle port) where it is absent.
Needs a checkout of the reference (LAB4D_REF_ROOT, default /root/reference); __graft_entry__.build() calls it."""
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(os.environ.get("LAB4D_REF_ROOT") or "/root/reference", "lab4d")
DST = os.path.join(ROOT, "oracle", "_ref")


def make(force=False):
    if not os.path.isdir(SRC):
        return os.path.isdir(os.path.join(DST, "lab4d"))
    dst = os.path.join(DST, "lab4d")
    if os.path.isdir(dst) and not force:
        return True
    os.makedirs(DST, exist_ok=True)
    shutil.rmtree(dst, ignore_errors=True)
    shutil.copytree(SRC, dst, ignore=shutil.ignore_patterns("__pycache__", "*.pyc", "build", "*.so"))
    return True


if __name__ == "__main__":
    print("oracle/_ref ready" if make(force="--force" in sys.argv) else "reference not available")
