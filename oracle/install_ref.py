"""Install the UNMODIFIED reference package under oracle/_ref (git-ignored build product, made by build() and kept
with the tree, so that the machine that runs the tests needs no copy of the reference's source).  Test / benchmark
infrastructure: nothing under theia_b200/ imports it.

    python -m pip install --no-index --no-build-isolation --no-deps --target oracle/_ref <copy of the reference>

(--no-deps: the reference pins tensorflow / hydra / a webdataset fork that the model classes do not need; the
install is done from a temporary copy because the reference's source tree may be read-only.)"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.path.join(HERE, "_ref")
SRC = "/root/reference"


def present() -> bool:
    return os.path.exists(os.path.join(REF, "theia", "models", "rvfm.py"))


def ensure(force: bool = False) -> bool:
    """True when oracle/_ref holds the reference package (installing it if the source tree is available)."""
    if present() and not force:
        return True
    if not os.path.exists(os.path.join(SRC, "pyproject.toml")):
        return False
    tmp = tempfile.mkdtemp(prefix="theia_ref_src_")
    try:
        src = os.path.join(tmp, "reference")
        shutil.copytree(SRC, src, ignore=shutil.ignore_patterns("media", ".git"))
        for d, _, files in os.walk(src):  # copytree keeps read-only modes; the wheel build writes into the copy
            os.chmod(d, 0o755)
            for f in files:
                os.chmod(os.path.join(d, f), 0o644)
        if os.path.isdir(REF):
            shutil.rmtree(REF)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps",
               "--target", REF, src]
        r = subprocess.run(cmd, capture_output=True, text=True, cwd=tmp)
        if r.returncode != 0:
            raise RuntimeError("pip install of the reference failed:\n" + r.stdout[-2000:] + r.stderr[-2000:])
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    return present()


if __name__ == "__main__":
    print("oracle/_ref present:", ensure(force="--force" in sys.argv))
