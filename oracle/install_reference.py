"""Installs the UNMODIFIED reference (pyDcop) into oracle/_ref/.  TEST INFRASTRUCTURE ONLY.

    python oracle/install_reference.py            (__graft_entry__.build() calls install())

The source tree is PYDCOP_REFERENCE, else /root/reference.  It is installed offline with
`pip install --no-index --no-deps --target oracle/_ref` from a temporary copy (the source tree may be
read-only), and its tests/instances data files are copied next to it.  oracle/_ref/ is git-ignored; once
built it is self-contained, so the tests, and bench.py's thread-mode baseline, use it on machines that
have no source tree (oracle/ref_shim.py).  Nothing in the product path imports it.  Without a source
tree and without an earlier install this does nothing, and the tests that need the reference skip.
"""
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCE = os.environ.get("PYDCOP_REFERENCE") or "/root/reference"
TARGET = os.path.join(HERE, "_ref")


def installed() -> bool:
    return (os.path.isdir(os.path.join(TARGET, "pydcop"))
            and os.path.isdir(os.path.join(TARGET, "tests", "instances")))


def install() -> bool:
    """True when oracle/_ref/ holds the reference afterwards."""
    if installed():
        return True
    if not os.access(os.path.join(SOURCE, "pydcop"), os.R_OK | os.X_OK):
        return False
    with tempfile.TemporaryDirectory() as td:
        cp = os.path.join(td, "ref")
        shutil.copytree(SOURCE, cp, ignore=shutil.ignore_patterns(".git", "__pycache__", "docs"))
        r = subprocess.run([sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
                            "--no-cache-dir", "--target", TARGET, "--upgrade", cp],
                           capture_output=True, text=True)
    if r.returncode != 0:
        print("reference install into oracle/_ref failed: " + r.stderr[-400:], file=sys.stderr)
        return False
    shutil.copytree(os.path.join(SOURCE, "tests", "instances"), os.path.join(TARGET, "tests", "instances"),
                    dirs_exist_ok=True)
    return installed()


if __name__ == "__main__":
    print(TARGET if install() else "no reference installed")
