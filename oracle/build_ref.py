"""Recipe for oracle/_ref: a byte-for-byte copy of the reference's OWN Python package, made from a checkout of
fabiojbg/LLMApiGateway next to this repository (`../reference`, or the directory LGW_REFERENCE_DIR names).  TEST INFRASTRUCTURE.

The reference (fabiojbg/LLMApiGateway) is pure Python, so "building" it is copying it.  oracle/_ref/ is git-ignored (no
reference source enters the history); where it exists, bench.py's CPU legs run the reference's real make_llm_request /
ChunkProcessorThread (oracle/ref_arm.py) next to the GPU numbers.  __graft_entry__.build() calls this; without a readable
reference checkout it keeps whatever oracle/_ref already holds.
"""
from __future__ import annotations

import os
import shutil
from pathlib import Path

HERE = Path(__file__).resolve().parent
REF = Path(os.environ.get("LGW_REFERENCE_DIR") or HERE.parent.parent / "reference")
DST = HERE / "_ref"


def _readable(p: Path) -> bool:
    try:
        return p.is_dir() and os.access(p, os.R_OK | os.X_OK)
    except OSError:                                 # e.g. a parent directory this user may not enter
        return False


def build() -> bool:
    """Refresh oracle/_ref from the reference checkout.  False when there is none and no oracle/_ref either."""
    if not _readable(REF / "llm_gateway_core"):
        return DST.is_dir()
    if DST.exists():
        shutil.rmtree(DST)
    DST.mkdir(parents=True)
    shutil.copytree(REF / "llm_gateway_core", DST / "llm_gateway_core", ignore=shutil.ignore_patterns("__pycache__", "*.pyc", "*.db"))
    for name in ("main.py", "requirements.txt", "pyproject.toml", "LICENSE"):
        if (REF / name).exists():
            shutil.copy2(REF / name, DST / name)
    (DST / "README.txt").write_text("Unmodified copy of fabiojbg/LLMApiGateway made by oracle/build_ref.py; not tracked by git.\n")
    return True


if __name__ == "__main__":
    print("oracle/_ref", "ready" if build() else "unavailable")
