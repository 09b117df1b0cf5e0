"""Installs the unmodified upstream ``pytensor-federated`` package into ``oracle/_ref`` (git-ignored).

The reference arm of the benchmark (``bench.py --impl reference``, ``baseline/reference_arm.py``) runs that
package through its own public API.  The package is pure Python, so installing it means laying its package
directory out under ``oracle/_ref``, as ``pip install --no-deps --target`` would.  pip itself is not used
because it builds inside the source checkout (``build/``, ``*.egg-info``, and the upstream ``setup.py``
writes ``py.typed`` into the package), which fails on a read-only checkout.

The source is the checkout named by ``$PYTENSOR_FEDERATED_SRC`` (default ``/root/reference``).  Only the
upstream release this repository was compared against is installed: ``michaelosthege/pytensor-federated`` at
commit 048212d (version 1.0.2), identified by the digest of its package files.  Without that checkout
nothing is installed and the reference arm reports itself unavailable.

    python oracle/build_reference.py
"""
from __future__ import annotations

import hashlib
import os
import shutil
import sys
from pathlib import Path
from typing import List, Optional

ROOT = Path(__file__).resolve().parent.parent
TARGET = ROOT / "oracle" / "_ref"
PACKAGE = "pytensor_federated"
DEFAULT_SOURCE = "/root/reference"
DIGEST = "ca77f270d3e1201e8b84cfb2daa2b13eaff49545b313ee8fa33eaf06d5c4b4f8"


def package_files(pkg: Path) -> List[Path]:
    """Every file of the package, relative to it, sorted (bytecode caches excluded)."""
    files = []
    for dirpath, dirnames, filenames in os.walk(pkg):
        dirnames[:] = [d for d in dirnames if d != "__pycache__"]
        files += [Path(dirpath, f).relative_to(pkg) for f in filenames if not f.endswith(".pyc")]
    return sorted(files)


def digest(pkg: Path) -> str:
    h = hashlib.sha256()
    for rel in package_files(pkg):
        h.update(str(rel).encode() + b"\0")
        h.update((pkg / rel).read_bytes())
    return h.hexdigest()


def install(source: Optional[str] = None) -> Optional[Path]:
    """Copies the upstream package to ``oracle/_ref/pytensor_federated``; returns that path, or None when the
    upstream checkout is missing, unreadable or not the pinned release."""
    pkg = Path(source or os.environ.get("PYTENSOR_FEDERATED_SRC") or DEFAULT_SOURCE) / PACKAGE
    try:
        if not package_files(pkg):   # os.walk reports a missing or unreadable directory as empty
            raise FileNotFoundError(f"no readable package at {pkg}")
        found = digest(pkg)
    except OSError as ex:
        print(f"oracle: upstream {PACKAGE} not installed ({ex})", file=sys.stderr)
        return None
    if found != DIGEST:
        print(f"oracle: {pkg} is not the pinned upstream release (digest {found}); not installed", file=sys.stderr)
        return None
    shutil.rmtree(TARGET, ignore_errors=True)
    for rel in package_files(pkg):
        dst = TARGET / PACKAGE / rel
        dst.parent.mkdir(parents=True, exist_ok=True)
        shutil.copyfile(pkg / rel, dst)   # contents only: the checkout may be read-only, the copy must not be
    assert digest(TARGET / PACKAGE) == DIGEST
    return TARGET / PACKAGE


if __name__ == "__main__":
    print(install(sys.argv[1] if len(sys.argv) > 1 else None))
