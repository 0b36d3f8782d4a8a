"""TEST / MEASUREMENT INFRASTRUCTURE — not part of the product path.

Recipe that makes the UNMODIFIED reference (microsoft/aurora, pure Python, `/root/reference/aurora`) importable on
the GPU box, where `/root/reference` does not exist:

    python oracle/build_ref.py            # build container only

* copies the reference's package directory `aurora/` byte for byte into `oracle/_ref/aurora/` — the reference's
  wheel is a pure-Python wheel (hatchling, `pyproject.toml:1-3`), i.e. installing it IS this copy; hatchling is not
  in this image, so `pip install --target` cannot run;
* adds the 4-symbol `timm` stand-in the reference needs to import (`tests/_shims/timm`, OUR code: `to_2tuple`,
  `to_3tuple`, `DropPath`, `trunc_normal_`; the real timm supplies no run-time arithmetic, SURVEY F4);
* writes `oracle/_ref/MANIFEST.json` with a SHA-256 per copied file, so that a run on the GPU box can state which
  reference bytes it timed / compared against.

`oracle/_ref/` is git-ignored (no reference source ever enters the history) but NOT gpurun-ignored, so it travels
to the GPU box like the built `.so`.  Only `tests/`, `bench.py`'s reference legs and `__graft_entry__.smoke()` may
import it (through `oracle/ref.py`).
"""

from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
REFERENCE = Path("/root/reference")
OUT = HERE / "_ref"


def _sha(path: Path) -> str:
    return hashlib.sha256(path.read_bytes()).hexdigest()


def reference_present() -> bool:
    """Whether the reference checkout can be read by this user (a stat() of a path it cannot traverse would raise)."""
    return os.access(REFERENCE / "aurora", os.R_OK | os.X_OK)


def build(force: bool = False) -> Path:
    src = REFERENCE / "aurora"
    if not reference_present():
        if (OUT / "aurora" / "__init__.py").exists():
            return OUT  # GPU box: use what travelled with the snapshot
        raise FileNotFoundError(f"{src} not found and {OUT} was not built; run oracle/build_ref.py in the build container")
    manifest_path = OUT / "MANIFEST.json"
    files = sorted(p for p in src.rglob("*") if p.is_file() and "__pycache__" not in p.parts)
    want = {str(p.relative_to(REFERENCE)): _sha(p) for p in files}
    if not force and manifest_path.exists():
        have = json.loads(manifest_path.read_text()).get("files", {})
        if have == want and (OUT / "timm" / "__init__.py").exists():
            return OUT
    if OUT.exists():
        shutil.rmtree(OUT)
    OUT.mkdir(parents=True)
    shutil.copytree(src, OUT / "aurora", ignore=shutil.ignore_patterns("__pycache__"))
    shutil.copytree(ROOT / "tests" / "_shims" / "timm", OUT / "timm", ignore=shutil.ignore_patterns("__pycache__"))
    for rel, digest in want.items():
        assert _sha(OUT / rel) == digest, rel
    manifest_path.write_text(json.dumps({
        "source": str(src), "what": "byte-for-byte copy of the reference package (pure-Python wheel contents)",
        "timm": "4-symbol stand-in from tests/_shims/timm (not reference code)", "files": want}, indent=1))
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv))
