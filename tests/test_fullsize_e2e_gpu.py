"""End-to-end parity at BASELINE.json's FULL configurations: the whole `forward` of the production models on the
production grids — 48 Swin blocks at D = 512 ... 2048, the fp16 encoder / decoder on physically scaled 13-level inputs,
the decoder's 842 400-row GEMMs — against the UNMODIFIED reference running in fp32 (no TF32) on a B200 with the same
parameters and the same Batch.  This is the reference's own acceptance test (`tests/test_model.py:27-86`) moved to the
benchmarked configurations.

The reference's outputs are stored in tests/golden/fullsize_<case>.npz (written by make_golden.py on a B200): its fp32
values at a fixed sample of points of every output field and of the backbone output, mean |fp32| over every whole field,
and the spread of its own bf16 recipe (`Aurora(autocast=True)`, aurora.py:327-343), rel-mean-abs against fp32 over every
whole field.  Our error is measured at the stored points.

Tolerance, per variable, rel-mean-abs error mean|out - ref| / mean|ref|:
    err(ours vs reference fp32)  <=  max( REF_TOL[var],  1.5 x err(reference autocast=True vs reference fp32) )
`REF_TOL` is the reference's own per-variable budget (1e-4 for 2t / msl / t / z, 5e-3 for the rest, `tests/fixtures.py`).
The second term states the claim precisely: our bf16 path must sit inside the spread of the reference's OWN bf16 recipe
measured on the very same inputs — at 48 blocks that recipe itself can leave the tight 1e-4 budget, which was written
for the 20-block small model in float64.  Both errors are printed.

A stage-level tap is compared too: the backbone output (what `Perceiver3DDecoder` consumes) of the reference, captured
with a forward hook, against the engine's decoder input buffer."""

import gc
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import fixtures as fx

pytestmark = pytest.mark.gpu
DEV = "cuda"
GOLD = Path(__file__).parent / "golden"
SEED = 5

CASES = {
    # name: bench workload (model class, grid, levels)
    "aurora_1p3b_0p25deg": "aurora-0.25deg-721x1440x13L",
    "aurora_small_0p25deg": "aurora-small-0.25deg-721x1440x13L",
    "aurora_airpollution_0p4deg": "aurora-airpollution-0.4deg-451x900x13L",
    "aurora_highres_0p1deg": "aurora-highres-0.1deg-1801x3600x13L",
}


def make_inputs(name):
    """The case's model with bench.py's random parameters (seed 5) on the device, and its Batch on the device."""
    import aurora_b200 as ab
    import bench

    cls, h, w, levels = bench.WORKLOADS[CASES[name]]
    model = getattr(ab, cls)(_init="empty", autocast=True).to(DEV).eval()
    bench.randomise_parameters_(model, seed=SEED)
    host = bench.make_host_batch(model.config, h, w, levels, pinned=False, seed=SEED)
    return model, host.to(DEV)


def run_ours(name):
    """Our forward of the case: {(group, var): output on the device}, the backbone output tap, the metadata."""
    model, dev_batch = make_inputs(name)
    pred = model.forward(dev_batch)
    torch.cuda.synchronize()
    ours = {("surf", k): v.clone() for k, v in pred.surf_vars.items()}
    ours.update({("atmos", k): v.clone() for k, v in pred.atmos_vars.items()})
    tap = next(t for (nm, _, _), t in model._engine._buf.items() if nm == "bb.concat").float().clone()
    meta = pred.metadata
    del pred
    model._engine = None
    del model
    gc.collect()
    torch.cuda.empty_cache()
    return ours, tap, meta


def sampled_rel(out: torch.Tensor, gold, group: str, row: int) -> float:
    """rel-mean-abs error of `out` against field `row` of `group` at the stored points: mean over the sample of
    |out - ref|, over the stored mean |ref| of the whole field."""
    idx = torch.from_numpy(gold[f"{group}.idx"].astype(np.int64)).to(out.device)
    got = out.reshape(-1)[idx].double().cpu()
    ref = torch.from_numpy(gold[f"{group}.val"][row]).double()
    return ((got - ref).abs().mean() / float(gold[f"{group}.absmean"][row])).item()


@pytest.mark.parametrize("name", sorted(CASES))
def test_full_size_forward_matches_the_unmodified_reference(name):
    gold = np.load(GOLD / f"fullsize_{name}.npz")
    ours, tap_ours, meta = run_ours(name)
    assert meta.time[0].timestamp() == float(gold["meta.time0"]) and meta.rollout_step == int(gold["meta.rollout_step"])
    assert tuple(meta.atmos_levels) == tuple(gold["meta.atmos_levels"].tolist())

    names = {grp: gold[f"{grp}.names"].tolist() for grp in ("surf", "atmos")}
    assert sorted(ours) == sorted((grp, k) for grp, ks in names.items() for k in ks)
    failures = []
    print(f"\n[full-size parity] {name} ({CASES[name]})")
    assert tap_ours.numel() == int(np.prod(gold["tap.shape"]))  # B = 1: the reference's tap is batch row 0
    tap_err = sampled_rel(tap_ours, gold, "tap", 0)
    tap_ref = float(gold["tap.spread"][0])
    print(f"  backbone output tap: ours {tap_err:.3e}   reference autocast {tap_ref:.3e}")
    for key in sorted(ours):
        grp, k = key
        row = names[grp].index(k)
        o = ours[key]
        assert tuple(o.shape) == tuple(gold[f"{grp}.shape"]) and torch.isfinite(o).all(), key
        e = sampled_rel(o, gold, grp, row)
        e_ref = float(gold[f"{grp}.spread"][row])
        bound = max(fx.tol_for(k), 1.5 * e_ref)
        print(f"  {grp:5s} {k:6s} ours {e:.3e}   reference autocast {e_ref:.3e}   bound {bound:.1e}"
              f"   {'(within the tight per-variable budget)' if e <= fx.tol_for(k) else ''}")
        if not e <= bound:
            failures.append((key, e, bound))
    assert not failures, failures
    assert tap_err <= max(5e-3, 1.5 * tap_ref), (tap_err, tap_ref)
