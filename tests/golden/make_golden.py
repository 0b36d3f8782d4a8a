"""Generate the golden fixtures in this directory by running the UNMODIFIED reference
(a checkout of microsoft/aurora, imported through the 4-symbol timm stand-in in tests/_shims) on the
deterministic inputs of tests/fixtures.py:

    PYTHONPATH=<reference checkout>:tests/_shims:. python tests/golden/make_golden.py [what ...]

`fullsize` needs a B200; `oracle/_ref` (made by oracle/build_ref.py) holds the reference and the stand-in:

    PYTHONPATH=oracle/_ref:. python tests/golden/make_golden.py fullsize

Outputs
    windows.npz        gather indices and mask group ids of roll->pad->window_partition_3d and
                       compute_3d_shifted_window_mask for the shape cases of SURVEY.md App. A.5
    windows_random.json  SHA-256 digests of the same maps on the random geometries of test_windows_random_cpu.py
    model_<case>.npz   float32 copies of the reference's float64 forward outputs (+ encoder / backbone taps)
    keys.json          state_dict key -> shape for the reference presets (parameter-layout parity)
    batch_reference.json, regrid_reference.npz   the reference's `Batch` transforms (test_batch_host.py)
    fullsize_<case>.npz  the reference's full-size forwards on a B200, sampled (test_fullsize_e2e_gpu.py)
"""

import dataclasses
import gc
import hashlib
import json
import math
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))

import aurora  # noqa: E402  (the reference)
from aurora.model import swin3d as ref_swin  # noqa: E402
from aurora.model.util import maybe_adjust_windows  # noqa: E402

from tests import fixtures as fx  # noqa: E402

WINDOW_CASES = [
    # (res, shifted)
    ((4, 45, 90), True), ((4, 45, 90), False), ((4, 4, 8), True), ((4, 4, 8), False),
    ((4, 15, 30), True), ((4, 15, 30), False), ((4, 38, 75), True), ((4, 38, 75), False),
    ((4, 12, 24), True), ((4, 12, 24), False), ((6, 13, 25), True), ((6, 13, 25), False),
    ((4, 8, 16), True), ((4, 2, 4), True), ((4, 1, 2), True), ((4, 90, 180), True), ((4, 75, 150), True),
]
# production shapes: only a checksum is stored
WINDOW_HASH_CASES = [((4, 180, 360), True), ((4, 180, 360), False), ((4, 150, 300), True), ((4, 90, 180), False)]
WS0 = (2, 6, 12)


def ref_window_maps(res, shifted, warped=True):
    c, h, w = res
    ss0 = tuple(s // 2 for s in WS0) if shifted else (0, 0, 0)
    ws, ss = maybe_adjust_windows(WS0, ss0, res)
    x = (torch.arange(c * h * w, dtype=torch.float64) + 1).view(1, c, h, w, 1)
    if not all(s == 0 for s in ss):
        x = torch.roll(x, shifts=(-ss[0], -ss[1], -ss[2]), dims=(1, 2, 3))
    pad = ((-c) % ws[0], (-h) % ws[1], (-w) % ws[2])
    x = ref_swin.pad_3d(x, pad)
    idx = ref_swin.window_partition_3d(x, ws).reshape(-1, ws[0] * ws[1] * ws[2]).long() - 1
    if all(s == 0 for s in ss):
        groups = None
    else:
        ref_swin.compute_3d_shifted_window_mask.cache_clear()
        mask, img = ref_swin.compute_3d_shifted_window_mask(c, h, w, ws, ss, torch.device("cpu"), torch.float32, warped)
        groups = ref_swin.window_partition_3d(img, ws).reshape(-1, ws[0] * ws[1] * ws[2]).to(torch.uint8)
        # the mask is fully determined by the group ids
        same = groups[:, :, None] == groups[:, None, :]
        assert torch.equal(mask, torch.where(same, 0.0, -100.0))
    return idx.numpy(), None if groups is None else groups.numpy()


def gen_windows():
    out = {}
    for res, shifted in WINDOW_CASES:
        for warped in (True, False):
            idx, g = ref_window_maps(res, shifted, warped)
            tag = f"{res[0]}x{res[1]}x{res[2]}_{'s' if shifted else 'u'}_{'w' if warped else 'n'}"
            out[f"idx_{tag}"] = idx.astype(np.int32)
            if g is not None:
                out[f"grp_{tag}"] = g
    hashes = {}
    for res, shifted in WINDOW_HASH_CASES:
        idx, g = ref_window_maps(res, shifted, True)
        tag = f"{res[0]}x{res[1]}x{res[2]}_{'s' if shifted else 'u'}_w"
        hashes[f"idx_{tag}"] = hashlib.sha256(idx.astype(np.int32).tobytes()).hexdigest()
        if g is not None:
            hashes[f"grp_{tag}"] = hashlib.sha256(g.astype(np.uint8).tobytes()).hexdigest()
    np.savez_compressed(HERE / "windows.npz", **out)
    (HERE / "windows_hashes.json").write_text(json.dumps(hashes, indent=1))
    print("windows.npz", len(out), "arrays;", len(hashes), "hashes")


from tests.golden.cases import MODEL_CASES  # noqa: E402


def build_reference(cfg_name, cls_name, seed):
    cfg = fx.CONFIGS[cfg_name]
    cls = getattr(aurora, cls_name)
    model = cls(**fx.model_kwargs(cfg, cls_name))
    extra = fx.air_extra_specs(cfg) if cls_name == "AuroraAirPollution" else ()
    sd = fx.make_state_dict(cfg, seed=seed, extra=extra)
    model.load_state_dict(sd, strict=True)  # also proves key/shape parity of aurora_b200.spec
    model.eval()
    return cfg, model, sd


def to_ref_batch(b):
    return aurora.Batch(
        surf_vars=dict(b.surf_vars), static_vars=dict(b.static_vars), atmos_vars=dict(b.atmos_vars),
        metadata=aurora.Metadata(lat=b.metadata.lat, lon=b.metadata.lon, time=b.metadata.time,
                                 atmos_levels=b.metadata.atmos_levels, rollout_step=b.metadata.rollout_step),
    )


def gen_models(only=None):
    for name, (cfg_name, cls_name, h, w, levels, bsz, step, seed) in MODEL_CASES.items():
        if only and not any(name.startswith(o) for o in only):
            continue
        cfg, model, _ = build_reference(cfg_name, cls_name, seed)
        batch = fx.case_inputs(MODEL_CASES[name])[2]
        taps = {}
        h1 = model.encoder.register_forward_hook(lambda m, i, o: taps.__setitem__("encoder", o.detach()))
        h2 = model.backbone.register_forward_hook(lambda m, i, o: taps.__setitem__("backbone", o.detach()))
        model = model.double()
        with torch.inference_mode():
            pred = model.forward(to_ref_batch(batch))
        h1.remove(), h2.remove()
        out = {f"surf.{k}": v.float().numpy() for k, v in pred.surf_vars.items()}
        out.update({f"atmos.{k}": v.float().numpy() for k, v in pred.atmos_vars.items()})
        out["tap.encoder"] = taps["encoder"].float().numpy()
        out["tap.backbone"] = taps["backbone"].float().numpy()
        out["meta.rollout_step"] = np.array(pred.metadata.rollout_step)
        out["meta.time0"] = np.array(pred.metadata.time[0].timestamp())
        np.savez_compressed(HERE / f"model_{name}.npz", **out)
        print(name, "ok", sum(v.nbytes for v in out.values()) // 1024, "KiB")


def gen_rollout():
    cfg, model, _ = build_reference("tiny_lora", "Aurora", 7)
    batch = fx.make_batch(cfg, 33, 64, levels=fx.LEVELS4, b=1, seed=7)
    out = {}
    with torch.inference_mode():
        for i, pred in enumerate(aurora.rollout(model.double(), to_ref_batch(batch), steps=3)):
            for k, v in pred.surf_vars.items():
                out[f"step{i}.surf.{k}"] = v.float().numpy()
            for k, v in pred.atmos_vars.items():
                out[f"step{i}.atmos.{k}"] = v.float().numpy()
            out[f"step{i}.rollout_step"] = np.array(pred.metadata.rollout_step)
    np.savez_compressed(HERE / "rollout_tiny_lora.npz", **out)
    print("rollout ok")


def gen_keys():
    keys = {}
    for cls_name in ("Aurora", "AuroraPretrained", "AuroraSmallPretrained", "Aurora12hPretrained", "AuroraHighRes",
                     "AuroraAirPollution", "AuroraWave"):
        m = getattr(aurora, cls_name)()
        keys[cls_name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    (HERE / "keys.json").write_text(json.dumps(keys))
    print("keys.json", {k: len(v) for k, v in keys.items()})


def gen_compat():
    """Published-layout checkpoints through the reference's `_adapt_checkpoint` of each model family."""
    from tests import compat_fixtures as cf

    out = {}
    for kind, cls_name in (("pretrained", "AuroraSmallPretrained"), ("air_pollution", "AuroraAirPollution"),
                           ("wave", "AuroraWave")):
        holder = types.SimpleNamespace(patch_size=cf.PATCH[kind])  # the adapters only read `self.patch_size`
        adapted = getattr(aurora, cls_name)._adapt_checkpoint(holder, cf.old_checkpoint(kind))
        out[kind] = cf.digest(adapted)
    (HERE / "compat.json").write_text(json.dumps(out, indent=0))
    print("compat.json", {k: len(v) for k, v in out.items()})


def gen_windows_random():
    """roll -> pad -> window_partition_3d and compute_3d_shifted_window_mask of the reference on the random geometries
    of test_windows_random_cpu.py, as digests of the arrays that test compares."""
    from tests import test_windows_random_cpu as T

    out = {}
    for chunk in range(T.REFERENCE_CHUNKS):
        recs = []
        for res, shifted, warped in T._geometries(30, 200 + chunk):
            c, h, w = res
            ss0 = tuple(s // 2 for s in WS0) if shifted else (0, 0, 0)
            ws, ss = maybe_adjust_windows(WS0, ss0, res)
            x = (torch.arange(c * h * w, dtype=torch.float64) + 1).view(1, c, h, w, 1)
            if any(ss):
                x = torch.roll(x, shifts=(-ss[0], -ss[1], -ss[2]), dims=(1, 2, 3))
            x = ref_swin.pad_3d(x, ((-c) % ws[0], (-h) % ws[1], (-w) % ws[2]))
            idx = ref_swin.window_partition_3d(x, ws).reshape(-1, ws[0] * ws[1] * ws[2]).long().numpy() - 1
            rec = {"res": list(res), "shifted": shifted, "warped": warped, "shift_after_adjust": any(ss),
                   "idx": fx.array_digest(idx.astype(np.int32))}
            if any(ss):
                ref_swin.compute_3d_shifted_window_mask.cache_clear()
                try:
                    mask, img = ref_swin.compute_3d_shifted_window_mask(c, h, w, ws, ss, torch.device("cpu"),
                                                                        torch.float32, warped)
                except RuntimeError:  # the reference's own `.view` fails on some degenerate grids (swin3d.py:355)
                    rec["mask"] = None
                else:
                    grp = ref_swin.window_partition_3d(img, ws).reshape(-1, ws[0] * ws[1] * ws[2]).to(torch.uint8)
                    same = grp[:, :, None] == grp[:, None, :]
                    assert fx.array_digest(mask) == fx.array_digest(torch.where(same, 0.0, -100.0)), res
                    rec["grp"], rec["mask"] = fx.array_digest(grp), fx.array_digest(mask)
            recs.append(rec)
        out[str(chunk)] = recs
    (HERE / "windows_random.json").write_text(json.dumps(out, indent=0))
    print("windows_random.json", sum(len(v) for v in out.values()), "geometries")


REGRID_SAMPLES = 256  # points per regridded field; the whole field enters through its sum


def gen_batch():
    """The reference's normalisation constants and `Batch` normalise / unnormalise / crop / regrid on the inputs of
    test_batch_host.py."""
    from aurora import normalisation as rn

    from tests import test_batch_host as T

    rb = to_ref_batch(T.transforms_batch())
    transforms = {"normalise": rb.normalise(surf_stats={}), "unnormalise": rb.normalise(surf_stats={}).unnormalise(surf_stats={}),
                  "crop3": rb.crop(3)}
    assert sorted(transforms) == sorted(T.batch_transforms(T.transforms_batch()))
    out = {"locations": {k: float(v) for k, v in rn.locations.items()},
           "scales": {k: float(v) for k, v in rn.scales.items()}, "transforms": {}}
    for name, b in transforms.items():
        rec = {"spatial_shape": list(b.spatial_shape), "lat": fx.array_digest(b.metadata.lat)}
        for grp in T.GROUPS:
            rec[grp] = {k: fx.array_digest(v) for k, v in getattr(b, grp).items()}
        out["transforms"][name] = rec
    (HERE / "batch_reference.json").write_text(json.dumps(out, indent=0))

    rng = np.random.Generator(np.random.PCG64(0))
    rb = to_ref_batch(T.regrid_batch())
    arrays = {}
    for res in T.REGRID_RES:
        b, tag = rb.regrid(res), T.regrid_tag(res)
        arrays[f"{tag}.spatial_shape"] = np.array(b.spatial_shape)
        arrays[f"{tag}.lat"], arrays[f"{tag}.lon"] = b.metadata.lat.numpy(), b.metadata.lon.numpy()
        for grp in T.GROUPS:
            g, fields = grp.split("_")[0], getattr(b, grp)
            arrays.update(sampled_fields(f"{tag}.{g}", fields, REGRID_SAMPLES, rng))
            arrays[f"{tag}.{g}.vmax"] = np.array([float(v.abs().max()) for v in fields.values()])
            arrays[f"{tag}.{g}.sum"] = np.array([float(v.double().sum()) for v in fields.values()])
    np.savez_compressed(HERE / "regrid_reference.npz", **arrays)
    print("batch_reference.json, regrid_reference.npz", len(arrays), "arrays")


def sampled_fields(prefix: str, fields: dict, n: int, rng) -> dict:
    """Fields of one shape at up to `n` fixed random points: `<prefix>.names`, `.shape`, `.idx` (sorted flat indices),
    `.val` (one row per field, float32)."""
    (shape,) = {tuple(v.shape) for v in fields.values()}
    assert math.prod(shape) < 2**31, shape
    idx = np.unique(rng.integers(0, math.prod(shape), n)).astype(np.int32)
    rows = [v.reshape(-1)[torch.from_numpy(idx).long().to(v.device)].float().cpu().numpy() for v in fields.values()]
    return {f"{prefix}.names": np.array(list(fields)), f"{prefix}.shape": np.array(shape), f"{prefix}.idx": idx,
            f"{prefix}.val": np.stack(rows)}


# points per field (2 KiB each): on a B200 the rel-mean-abs error at these points came within 20 % of the whole-field
# value for every field of the four cases, each at least a third inside its bound
FULLSIZE_SAMPLES = 512


def gen_fullsize(only=None):
    """The reference's full-size forwards for test_fullsize_e2e_gpu.py, on a B200: fp32 with TF32 off and its own
    autocast recipe, on that test's inputs.  Stores the fp32 outputs and backbone output at a fixed sample of points,
    mean |fp32| of every whole field and the spread autocast vs fp32 over every whole field; prints our error over the
    whole field next to the one at the stored points."""
    import bench
    from tests import test_fullsize_e2e_gpu as T

    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False  # conv3d patch embedding of the reference in true fp32
    rng = np.random.Generator(np.random.PCG64(0))
    for case in sorted(T.CASES):
        if only and not any(case.startswith(o) for o in only):
            continue
        ours, tap_ours = T.run_ours(case)[:2]
        ours[("tap", "backbone")] = tap_ours
        model, dev_batch = T.make_inputs(case)
        sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
        del model
        rb = to_ref_batch(dev_batch)
        runs = {}
        for tag, autocast in (("fp32", False), ("autocast", True)):
            with torch.device("cuda"):
                rmodel = getattr(aurora, bench.WORKLOADS[T.CASES[case]][0])(autocast=autocast)
            rmodel.load_state_dict(sd, strict=True)
            rmodel = rmodel.eval()
            taps = {}
            hook = rmodel.backbone.register_forward_hook(lambda m, i, o: taps.__setitem__("tap", o.detach().float()[0]))
            with torch.inference_mode():
                rp = rmodel.forward(rb)
            hook.remove()
            torch.cuda.synchronize()
            fields = {("surf", k): v for k, v in rp.surf_vars.items()}
            fields.update({("atmos", k): v for k, v in rp.atmos_vars.items()})
            fields[("tap", "backbone")] = taps["tap"]
            runs[tag] = fields, rp.metadata
            del rp, rmodel
            gc.collect()
            torch.cuda.empty_cache()
        ref, meta = runs["fp32"]
        out = {"meta.time0": np.array(meta.time[0].timestamp()), "meta.rollout_step": np.array(meta.rollout_step),
               "meta.atmos_levels": np.array(meta.atmos_levels)}
        print(f"[fullsize golden] {case}")
        for group in ("surf", "atmos", "tap"):
            fields = {k: v for (g, k), v in ref.items() if g == group}
            out.update(sampled_fields(group, fields, FULLSIZE_SAMPLES, rng))
            out[f"{group}.absmean"] = np.array([v.double().abs().mean().item() for v in fields.values()])
            out[f"{group}.spread"] = np.array([fx.rel_mean_abs(runs["autocast"][0][(group, k)], v) for k, v in fields.items()])
            for row, (k, v) in enumerate(fields.items()):
                whole = fx.rel_mean_abs(ours[(group, k)], v)
                print(f"  {group:5s} {k:8s} ours: whole field {whole:.3e}, at the stored points "
                      f"{T.sampled_rel(ours[(group, k)], out, group, row):.3e}   reference autocast {out[f'{group}.spread'][row]:.3e}")
        del runs, ref, ours
        gc.collect()
        torch.cuda.empty_cache()
        np.savez_compressed(HERE / f"fullsize_{case}.npz", **out)


if __name__ == "__main__":
    only = [a.split("=", 1)[1] for a in sys.argv[1:] if a.startswith("--only=")]  # model / full-size case name prefixes
    what = [a for a in sys.argv[1:] if not a.startswith("--only=")] or ["windows", "windows_random", "models", "rollout",
                                                                         "keys", "compat", "batch"]
    torch.manual_seed(0)
    if "windows" in what:
        gen_windows()
    if "windows_random" in what:
        gen_windows_random()
    if "batch" in what:
        gen_batch()
    if "fullsize" in what:
        gen_fullsize(only)
    if "models" in what:
        gen_models(only)
    if "rollout" in what:
        gen_rollout()
    if "keys" in what:
        gen_keys()
    if "compat" in what:
        gen_compat()
