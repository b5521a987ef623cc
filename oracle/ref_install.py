"""Installs the unmodified reference package (dgl-ke's python/ directory, KGE_REFERENCE_PY) under oracle/_ref, where
cpu_bench.py runs its own training step as the CPU baseline.  oracle/_ref is a build product, kept out of git."""
import os
import shutil
import subprocess
import sys
import tempfile

from ref_harness import REFERENCE_PY

REF_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def installed():
    return os.path.isdir(os.path.join(REF_DIR, "dglke"))


def install():
    """pip install --no-index --no-deps of a copy of the reference's python/ tree (the tree itself may be read-only).
    Skipped when the reference is absent or already installed; when the install fails the CPU baseline times the
    oracle port instead."""
    if installed() or not os.path.isdir(os.path.join(REFERENCE_PY, "dglke")):
        return
    tmp = tempfile.mkdtemp(prefix="dglke_ref_")
    try:
        shutil.copytree(REFERENCE_PY, os.path.join(tmp, "python"))
        subprocess.run([sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
                        "--target", REF_DIR, os.path.join(tmp, "python")],
                       check=False, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
