#!/usr/bin/env python
"""Install the UNMODIFIED reference into oracle/_ref/ so that bench.py can time its own CPU path
(oracle/_ref/ is git-ignored).  __graft_entry__.build() calls this with the checkout recorded as
`reference_path` in BASELINE.json; where that checkout is missing or unreadable it installs nothing.

The reference has no setup.py / pyproject.toml (its docs say `pip install SPART-python`, the tree is used
with PYTHONPATH=src), so a `pip install --target oracle/_ref <checkout>` recipe does not apply:
this script copies the package directory src/SPART -- Python sources and the pickled tables it loads at
run time -- byte for byte, plus the six-line `nvtx` stand-in the reference's hard `import nvtx`
(SPART.py:23) needs where the nvtx package is not installed.  Nothing is copied into tracked paths.

usage: python tools/install_reference.py [--src <reference checkout>]"""
import argparse
import filecmp
import json
import shutil
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
DEST = ROOT / "oracle" / "_ref"


def default_source():
    """The reference checkout BASELINE.json records."""
    return json.loads((ROOT / "BASELINE.json").read_text())["reference_path"]


def install(src=None, dest=DEST):
    """Copy src/SPART of the reference checkout `src` into `dest`; returns the copy, or None when there is no
    readable checkout at `src`."""
    pkg = Path(src or default_source()) / "src" / "SPART"
    try:
        if not pkg.is_dir():
            return None
    except OSError:          # a directory on the way this user may not read: no reference here
        return None
    dest = Path(dest)
    dest.mkdir(parents=True, exist_ok=True)
    target = dest / "SPART"
    if target.exists():
        shutil.rmtree(target)
    shutil.copytree(pkg, target, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    shutil.copyfile(ROOT / "tools" / "_nvtx_stub" / "nvtx.py", dest / "nvtx.py")
    cmp = filecmp.dircmp(pkg, target, ignore=["__pycache__"])
    assert not cmp.diff_files and not cmp.left_only, "reference copy differs from its source"
    (dest / "INSTALLED_FROM").write_text(f"{pkg}\n")
    return target


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default=None, help="reference checkout (default: BASELINE.json reference_path)")
    t = install(ap.parse_args().src)
    print("installed" if t else "no reference tree found", t or "")
    sys.exit(0 if t else 1)
