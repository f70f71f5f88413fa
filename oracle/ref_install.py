"""Copy the unmodified mbrl-lib package into ``oracle/_ref/`` (git-ignored), where the tests and bench.py's reference
arm import it from (``baseline/reference_arm.py``).

mbrl-lib is pure Python, so installing it is a copy of its ``mbrl`` package; the four pure-Python dependencies it
imports at module level are stood in for by ``oracle/ref_shims``.  The source tree is ``$MBRL_LIB_SRC`` or else the
``reference_path`` recorded in ``BASELINE.json``.  Where neither is readable an existing copy is kept as it is, and
without one the tests that need mbrl-lib's own code skip.
"""
from __future__ import annotations

import json
import os
import shutil
from typing import Optional

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def source_tree() -> str:
    src = os.environ.get("MBRL_LIB_SRC")
    if src:
        return src
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        return json.load(f)["reference_path"]


def install(src: Optional[str] = None) -> Optional[str]:
    """Copy ``<src>/mbrl`` to ``oracle/_ref/mbrl``; returns the copy's directory, or None when ``src`` has no package."""
    pkg = os.path.join(src or source_tree(), "mbrl")
    if not os.path.isfile(os.path.join(pkg, "__init__.py")):
        return None
    dst = os.path.join(REF_DIR, "mbrl")
    tmp = dst + ".tmp"
    shutil.rmtree(tmp, ignore_errors=True)
    shutil.copytree(pkg, tmp, ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    shutil.rmtree(dst, ignore_errors=True)
    os.replace(tmp, dst)
    return dst
