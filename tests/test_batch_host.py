"""`Batch` / `Metadata` host logic (no GPU): validation and error behaviour of `aurora/batch.py:24-190`, the
normalisation constants of `aurora/normalisation.py`, and normalise / unnormalise / crop / regrid against what the
reference classes computed on the same inputs (tests/golden/batch_reference.json and regrid_reference.npz, written by
make_golden.py)."""

import json
from datetime import datetime
from pathlib import Path

import numpy as np
import pytest
import torch

from aurora_b200 import Batch, Metadata
from aurora_b200 import stats
from tests import fixtures as fx

GOLD = Path(__file__).parent / "golden"
GROUPS = ("surf_vars", "static_vars", "atmos_vars")


def _meta(h=17, w=32, **kw):
    base = dict(lat=torch.linspace(90, -90, h), lon=torch.linspace(0, 360, w + 1)[:-1],
                time=(datetime(2020, 6, 1, 12, 0),), atmos_levels=(100, 250, 500, 850))
    base.update(kw)
    return Metadata(**base)


@pytest.mark.parametrize("kw,msg", [
    (dict(lat=torch.linspace(91, -90, 17)), "Latitudes must be in the range"),
    (dict(lon=torch.linspace(0, 360, 32)), "Longitudes must be in the range"),
    (dict(lat=torch.linspace(-90, 90, 17)), "strictly decreasing"),
    (dict(lon=torch.linspace(0, 360, 33)[:-1].flip(0)), "strictly increasing"),
    (dict(lat=torch.linspace(90, -90, 17)[:, None].expand(17, 32)), "both be vectors or both be matrices"),
])
def test_metadata_validation_errors(kw, msg):
    with pytest.raises(ValueError, match=msg):
        _meta(**kw)


def test_crop_drops_one_latitude_row_and_rejects_more():
    cfg = fx.CONFIGS["tiny"]
    b = fx.make_batch(cfg, 17, 32, levels=fx.LEVELS4)
    c = b.crop(4)
    assert c.spatial_shape == (16, 32) and c.metadata.lat.shape == (16,)
    assert torch.equal(c.surf_vars["2t"], b.surf_vars["2t"][..., :-1, :])
    assert torch.equal(c.atmos_vars["t"], b.atmos_vars["t"][..., :-1, :])
    assert torch.equal(c.static_vars["z"], b.static_vars["z"][:-1])
    assert c.crop(4) is c  # already a multiple: unchanged
    with pytest.raises(ValueError, match="at most be one latitude too many"):
        fx.make_batch(cfg, 18, 32, levels=fx.LEVELS4).crop(4)
    with pytest.raises(ValueError, match="Width"):
        fx.make_batch(cfg, 16, 30, levels=fx.LEVELS4).crop(4)


def test_normalise_roundtrip_and_overrides():
    cfg = fx.CONFIGS["tiny"]
    b = fx.make_batch(cfg, 16, 32, levels=fx.LEVELS4)
    n = b.normalise()
    loc, sc = stats.surf_stats_of("2t")
    assert torch.allclose(n.surf_vars["2t"], (b.surf_vars["2t"] - loc) / sc)
    locs, scs = stats.atmos_stats_of("q", fx.LEVELS4)
    want = (b.atmos_vars["q"] - torch.tensor(locs)[:, None, None]) / torch.tensor(scs)[:, None, None]
    assert torch.allclose(n.atmos_vars["q"], want)
    back = n.unnormalise()
    for k in b.surf_vars:
        assert torch.allclose(back.surf_vars[k], b.surf_vars[k], rtol=1e-5, atol=1e-5 * abs(stats.surf_stats_of(k)[0]))
    over = {"2t": (1.0, 2.0)}
    assert torch.allclose(b.normalise(surf_stats=over).surf_vars["2t"], (b.surf_vars["2t"] - 1.0) / 2.0)
    d = b.type(torch.float64)
    assert d.surf_vars["2t"].dtype == d.metadata.lat.dtype == torch.float64
    assert stats.level_to_str(850) == "850" and stats.level_to_str(12.5) == "12_5"


def batch_transforms(b):
    """The transforms of `test_against_reference_classes_live`, by the name they are stored under."""
    return {"normalise": b.normalise(), "unnormalise": b.normalise().unnormalise(), "crop3": b.crop(3)}


def transforms_batch():
    return fx.make_batch(fx.CONFIGS["tiny_air"], 46, 90, levels=fx.LEVELS13, b=2)


def test_against_reference_classes_live():
    gold = json.loads((GOLD / "batch_reference.json").read_text())
    # every normalisation constant of the reference is in our table, bit for bit as float64
    assert stats.locations == gold["locations"]
    assert stats.scales == gold["scales"]
    for name, ours in batch_transforms(transforms_batch()).items():
        ref = gold["transforms"][name]
        assert list(ours.spatial_shape) == ref["spatial_shape"], name
        for grp in GROUPS:
            assert list(getattr(ours, grp)) == list(ref[grp]), (name, grp)
            for k, digest in ref[grp].items():
                assert fx.array_digest(getattr(ours, grp)[k]) == digest, (name, grp, k)
        assert fx.array_digest(ours.metadata.lat) == ref["lat"], name


def test_regrid_properties():
    """Bilinear re-gridding (aurora/batch.py:192-222): a field that is linear in latitude and piecewise linear in
    longitude is reproduced exactly, re-gridding to the same grid is the identity, shapes follow the reference."""
    cfg = fx.CONFIGS["tiny"]
    b = fx.make_batch(cfg, 17, 32, levels=fx.LEVELS4)          # 11.25-degree grid including both poles
    same = b.regrid(11.25)
    assert same.spatial_shape == (17, 32)
    for k in b.surf_vars:
        assert torch.allclose(same.surf_vars[k], b.surf_vars[k], rtol=5e-6, atol=1e-4)
    fine = b.regrid(5.625)
    assert fine.spatial_shape == (33, 64) and fine.atmos_vars["t"].shape == (1, 2, 4, 33, 64)
    assert fine.metadata.lat.dtype == torch.float64 and float(fine.metadata.lat[0]) == 90.0 and float(fine.metadata.lon[-1]) < 360
    lat, lon = b.metadata.lat.double(), b.metadata.lon.double()
    ramp = (3.0 * lat[:, None] + 0.0 * lon[None, :]).float()
    bb = Batch({"2t": ramp[None, None]}, {"z": ramp}, {"t": ramp[None, None, None]}, b.metadata)
    out = bb.regrid(5.625)
    want = (3.0 * out.metadata.lat[:, None] + 0.0 * out.metadata.lon[None, :]).float()
    assert torch.allclose(out.static_vars["z"], want, atol=1e-4)
    # every second point of the finer grid is an original grid point
    assert torch.allclose(fine.surf_vars["2t"][..., ::2, ::2], b.surf_vars["2t"], rtol=5e-6, atol=1e-4)


REGRID_RES = (5.0, 11.25, 7.3)


def regrid_tag(res: float) -> str:
    return str(res).replace(".", "p")


def regrid_batch():
    return fx.make_batch(fx.CONFIGS["tiny"], 17, 32, levels=fx.LEVELS4, b=2)


@pytest.mark.parametrize("res", REGRID_RES)
def test_regrid_against_reference_live(res):
    """The reference's regridded fields are stored at a fixed sample of points, with their max |value| and their sum:
    every stored point within the tolerance below, and the sum over the whole field within the sum of those bounds."""
    gold = np.load(GOLD / "regrid_reference.npz")
    tag = regrid_tag(res)
    ours = regrid_batch().regrid(res)
    assert list(ours.spatial_shape) == gold[f"{tag}.spatial_shape"].tolist()
    assert torch.allclose(ours.metadata.lat, torch.from_numpy(gold[f"{tag}.lat"]), atol=1e-12)
    assert torch.allclose(ours.metadata.lon, torch.from_numpy(gold[f"{tag}.lon"]), atol=1e-12)
    for grp in GROUPS:
        g, fields = grp.split("_")[0], getattr(ours, grp)
        names = gold[f"{tag}.{g}.names"].tolist()
        assert sorted(names) == sorted(fields), grp
        idx = torch.from_numpy(gold[f"{tag}.{g}.idx"].astype(np.int64))
        for row, k in enumerate(names):
            got = fields[k]
            assert got.dtype == torch.float32 and list(got.shape) == gold[f"{tag}.{g}.shape"].tolist(), (grp, k)
            v = torch.from_numpy(gold[f"{tag}.{g}.val"][row])
            vmax = float(gold[f"{tag}.{g}.vmax"][row])
            atol, rtol = 1e-6 * vmax, 2e-6
            sample = got.reshape(-1)[idx]
            assert torch.allclose(sample, v, rtol=rtol, atol=atol), (grp, k, float((sample - v).abs().max()))
            total = float(got.double().sum()) - float(gold[f"{tag}.{g}.sum"][row])
            assert abs(total) <= got.numel() * (atol + rtol * vmax), (grp, k, total)


def test_netcdf_io_needs_xarray_like_the_reference(tmp_path):
    try:
        import xarray  # noqa: F401
    except ImportError:
        b = fx.make_batch(fx.CONFIGS["tiny"], 16, 32, levels=fx.LEVELS4)
        with pytest.raises(RuntimeError, match="`xarray` must be installed"):
            b.to_netcdf(tmp_path / "b.nc")
        with pytest.raises(RuntimeError, match="`xarray` must be installed"):
            Batch.from_netcdf(tmp_path / "b.nc")
        return
    b = fx.make_batch(fx.CONFIGS["tiny"], 16, 32, levels=fx.LEVELS4)   # round trip when the libraries are there
    b.to_netcdf(tmp_path / "b.nc")
    r = Batch.from_netcdf(tmp_path / "b.nc")
    for k in b.surf_vars:
        assert torch.equal(r.surf_vars[k], b.surf_vars[k])
    assert r.metadata.time == b.metadata.time and tuple(r.metadata.atmos_levels) == tuple(b.metadata.atmos_levels)
