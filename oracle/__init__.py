"""Test infrastructure: CPU restatements of the reference path (never imported by the product package).

`REFERENCE_ROOT` is a checkout of the original TextMAE-Image-Compression project, read by the cross-checks that execute
its code where it lies and by the scripts that regenerate tests/golden/: $TMAE_REFERENCE_DIR, else oracle/_ref/ (ignored
by git).  Without it those cross-checks skip; the goldens carry the reference outputs the rest of the suite compares with.
"""
from __future__ import annotations

import os
from pathlib import Path

REFERENCE_ROOT = Path(os.environ.get("TMAE_REFERENCE_DIR") or Path(__file__).resolve().parent / "_ref")
SKIP_REASON = "needs a checkout of the original project (TMAE_REFERENCE_DIR, or oracle/_ref)"


def reference_has(*rel: str) -> bool:
    """True when every `rel` file exists under REFERENCE_ROOT; a location this user cannot read counts as absent."""
    try:
        return all((REFERENCE_ROOT / r).is_file() for r in rel)
    except OSError:
        return False
