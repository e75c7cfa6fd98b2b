"""Install the UNMODIFIED reference hot-path packages into oracle/_ref (git-ignored build output of `build()`).

TEST / BENCH INFRASTRUCTURE.  The reference is not a pip project (no setup.py / pyproject.toml), so it cannot be pip-installed
as it lies.  This script copies its `pose_diffusion/models` and `pose_diffusion/util` -- byte for byte -- to a temporary
directory, puts a three-line setup.py beside them there, and lets pip install that into oracle/_ref.  Nothing is written into
the reference checkout, nothing of the reference enters the tracked repository.  `oracle/ref_loader.py` imports the modules from
oracle/_ref when the reference checkout itself is absent, which lets `bench.py --impl reference` time the reference's OWN
modules (`cpu_baseline.kind = "reference"`) on a machine that only received the built tree.

    python oracle/install_reference.py          # no-op when the reference checkout is absent or oracle/_ref is up to date
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE_ROOT = os.environ.get("POSEDIFF_REFERENCE_ROOT", "/root/reference")
TARGET = os.path.join(ROOT, "oracle", "_ref")
PACKAGES = ("models", "util")


def tree_digest(base: str) -> str:
    h = hashlib.sha256()
    for pkg in PACKAGES:
        for dirpath, dirnames, filenames in sorted(os.walk(os.path.join(base, pkg))):
            dirnames[:] = sorted(d for d in dirnames if d != "__pycache__")
            for name in sorted(filenames):
                if name.endswith(".py"):
                    path = os.path.join(dirpath, name)
                    h.update(os.path.relpath(path, base).encode())
                    h.update(open(path, "rb").read())
    return h.hexdigest()


def install(verbose: bool = True) -> str:
    """Returns 'absent' (no reference tree here), 'current' or 'installed'."""
    src = os.path.join(REFERENCE_ROOT, "pose_diffusion")
    if not os.path.isdir(os.path.join(src, "models")):
        return "absent"
    digest = tree_digest(src)
    stamp = os.path.join(TARGET, "REFERENCE_SHA256")
    if os.path.exists(stamp) and open(stamp).read().strip() == digest and tree_digest(TARGET) == digest:
        return "current"
    with tempfile.TemporaryDirectory(prefix="posediff_ref_") as tmp:
        for pkg in PACKAGES:
            shutil.copytree(os.path.join(src, pkg), os.path.join(tmp, pkg), ignore=shutil.ignore_patterns("__pycache__"))
        with open(os.path.join(tmp, "setup.py"), "w") as fh:
            fh.write("from setuptools import setup, find_packages\n"
                     "setup(name='posediffusion_reference_hotpath', version='0', packages=find_packages())\n")
        if os.path.isdir(TARGET):
            shutil.rmtree(TARGET)
        os.makedirs(TARGET, exist_ok=True)
        cmd = [sys.executable, "-m", "pip", "install", "--no-index", "--no-build-isolation", "--no-deps", "--target", TARGET, tmp]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("pip install of the reference copy failed:\n" + res.stdout + res.stderr)
    if tree_digest(TARGET) != digest:
        raise RuntimeError("oracle/_ref does not match the reference tree after the install")
    with open(stamp, "w") as fh:
        fh.write(digest + "\n")
    if verbose:
        print(f"installed the reference's models/ and util/ into {TARGET} (sha256 {digest[:16]})")
    return "installed"


if __name__ == "__main__":
    print(install())
