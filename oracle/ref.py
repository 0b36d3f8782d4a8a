"""TEST / MEASUREMENT INFRASTRUCTURE — not part of the product path.

Import the UNMODIFIED reference package from `oracle/_ref` (made by `oracle/build_ref.py`) and build reference
models / batches for the parity tests and for `bench.py`'s reference legs (`cpu_baseline`, `gpu_reference`,
`--impl reference`).  Nothing under `aurora_b200/` imports this module.
"""

from __future__ import annotations

import importlib
import sys
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
REF_DIR = HERE / "_ref"


def available() -> bool:
    from oracle import build_ref

    return (REF_DIR / "aurora" / "__init__.py").exists() or build_ref.reference_present()


def load():
    """The reference's top-level module (`import aurora`), imported from oracle/_ref."""
    if "aurora" in sys.modules and getattr(sys.modules["aurora"], "__file__", "").startswith(str(REF_DIR)):
        return sys.modules["aurora"]
    from oracle import build_ref

    build_ref.build()  # no-op when up to date; on the GPU box it only checks that the copy travelled
    if str(REF_DIR) not in sys.path:
        sys.path.insert(0, str(REF_DIR))
    for name in [m for m in sys.modules if m == "aurora" or m.startswith("aurora.") or m == "timm" or m.startswith("timm.")]:
        del sys.modules[name]  # a copy imported from /root/reference by another test: same bytes, but keep one origin
    return importlib.import_module("aurora")


def build_model(cls_name: str, state_dict: dict | None = None, device="cpu", **kwargs):
    """A reference model of class `cls_name` (e.g. "AuroraPretrained") in eval mode, optionally loaded with
    `state_dict` (strict)."""
    ref = load()
    model = getattr(ref, cls_name)(**kwargs)
    if state_dict is not None:
        model.load_state_dict(state_dict, strict=True)
    return model.to(device).eval()


def to_ref_batch(batch, device=None):
    """An `aurora_b200.Batch` (or anything with the same fields) as the reference's `aurora.Batch`, sharing the
    tensors (moved to `device` if given)."""
    ref = load()
    mv = (lambda t: t) if device is None else (lambda t: t.to(device))
    md = batch.metadata
    return ref.Batch(
        surf_vars={k: mv(v) for k, v in batch.surf_vars.items()},
        static_vars={k: mv(v) for k, v in batch.static_vars.items()},
        atmos_vars={k: mv(v) for k, v in batch.atmos_vars.items()},
        metadata=ref.Metadata(lat=mv(md.lat), lon=mv(md.lon), time=tuple(md.time), atmos_levels=tuple(md.atmos_levels),
                              rollout_step=md.rollout_step),
    )


@torch.inference_mode()
def forward(model, batch):
    return model.forward(batch)
