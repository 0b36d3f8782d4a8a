"""bench.py contract checks that need no GPU: the reference arm (the unmodified reference from oracle/_ref on the host
cores, or the oracle port where that copy was not built) prints ONE JSON line with the keys a consumer reads, on rank 0
only, and the ncu summariser parses a metrics CSV."""

import gzip
import json
import os
import subprocess
import sys
from pathlib import Path

from oracle import build_ref, ref

ROOT = Path(__file__).resolve().parent.parent


def _run(args, env=None):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=600,
                       env={**os.environ, **(env or {})}, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [ln for ln in r.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_prints_one_contract_line():
    lines = _run(["--impl", "reference", "--workload", "aurora-small-17x32x4L", "--steps", "2", "--warmup", "1"])
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "forecast-steps/sec" and d["unit"] == "forecast-steps/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    # `ms_per_step` is the wall time of one timed (bounded-sample) step — K of them fit in the run — and a whole forecast
    # step is `sample_scale` of them, the factor measured against ONE complete reference forward in the same run
    assert d["value"] > 0 and abs(d["ms_per_whole_step"] - 1000.0 / d["value"]) < 1e-6 * d["ms_per_whole_step"]
    assert abs(d["ms_per_step"] * d["sample_scale"] / d["ms_per_whole_step"] - 1.0) < 1e-6
    assert d["config"]["workload"] == "aurora-small-17x32x4L" and d["config"]["parallelism"] == "single GPU"
    cb = d["cpu_baseline"]
    assert cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb and cb["samples"] == 2
    # the unmodified reference when oracle/_ref was built (it needs the reference checkout), else the oracle port
    if ref.available():
        assert cb["kind"] == "reference" and cb["complete_forward_seconds"] > 0
    else:
        assert cb["kind"] == "port" and cb["sample_seconds_median"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_reference_arm_is_silent_on_other_ranks():
    assert _run(["--impl", "reference", "--workload", "aurora-small-17x32x4L", "--steps", "1", "--warmup", "1", "--gpus", "2"],
                env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_ncu_summariser_reads_the_committed_launch_csv(tmp_path):
    sys.path.insert(0, str(ROOT / "tools"))
    src = ROOT / "profiles" / "r01m_launches.csv.gz"
    csv_path = tmp_path / "launches.csv"
    csv_path.write_bytes(gzip.open(src).read())
    r = subprocess.run([sys.executable, str(ROOT / "tools" / "ncu_traffic.py"), str(csv_path), "--tag", "zz_pytest",
                        "--workload", "zz-test-workload"], capture_output=True, text=True, cwd=ROOT, timeout=300)
    try:
        assert r.returncode == 0, r.stderr[-2000:]
        md = (ROOT / "profiles" / "zz_pytest_launch_list.md").read_text()
        assert "gemm2_bf16_tn_kernel" in md and "window_attention_tc_kernel" in md
        rec = json.loads((ROOT / "profiles" / "gemm_traffic.json").read_text())
        assert 5e8 < rec["zz-test-workload"]["dram_bytes_per_launch"] < 8e8
    finally:
        for f in ("zz_pytest_launch_list.md", "zz_pytest_launches.csv.gz"):
            (ROOT / "profiles" / f).unlink(missing_ok=True)
        f = ROOT / "profiles" / "gemm_traffic.json"
        rec = json.loads(f.read_text())
        rec.pop("zz-test-workload", None)
        f.write_text(json.dumps(rec, indent=1) + "\n")


def test_both_arms_report_the_same_config_and_parallelism():
    """`config` is computed from the command line alone, so the driver sees identical dicts from `--impl ours` and
    `--impl reference`; `auto` shards a forecast by latitude whenever the grid allows and falls back to replicas otherwise."""
    sys.path.insert(0, str(ROOT))
    import bench

    for wl in bench.WORKLOADS:
        for n in (1, 2, 4, 8):
            assert bench.workload_config(wl, n, "auto") == bench.workload_config(wl, n, "auto")
    assert bench.resolve_parallelism("aurora-0.25deg-721x1440x13L", 8, "auto") == "latshard"
    assert bench.resolve_parallelism("aurora-0.25deg-721x1440x13L", 1, "auto") == "single GPU"
    assert bench.resolve_parallelism("aurora-0.25deg-721x1440x13L", 8, "replicas") == "replicas"
    # 150 token rows: an odd 2x2 merge inside the U-Net -> cannot be banded -> replicas (explicit `latshard` raises)
    assert bench.resolve_parallelism("aurora-airpollution-0.4deg-451x900x13L", 8, "auto") == "replicas"
    import pytest

    with pytest.raises(NotImplementedError):
        bench.resolve_parallelism("aurora-airpollution-0.4deg-451x900x13L", 8, "latshard")
    cfg = bench.workload_config("aurora-0.25deg-721x1440x13L", 8, "auto")
    assert cfg["workload"] == "aurora-0.25deg-721x1440x13L" and "latitude-sharded over 8" in cfg["parallelism"]


def test_reference_copy_matches_its_manifest():
    """oracle/_ref (the copy of the unmodified reference) is byte-for-byte what its manifest says, and — where the
    reference checkout is readable — what that checkout holds."""
    import hashlib

    copy = ROOT / "oracle" / "_ref"
    if not (copy / "MANIFEST.json").exists():
        import pytest

        pytest.skip("oracle/_ref not built")
    man = json.loads((copy / "MANIFEST.json").read_text())
    assert man["files"], "empty manifest"
    for rel, digest in man["files"].items():
        assert hashlib.sha256((copy / rel).read_bytes()).hexdigest() == digest, rel
        if build_ref.reference_present():
            assert hashlib.sha256((build_ref.REFERENCE / rel).read_bytes()).hexdigest() == digest, rel


def test_dump_outputs_is_capped_and_repeatable(tmp_path, monkeypatch):
    """`--dump-outputs`: one float32 .npy per predicted field; over the size cap every field is a sample of its own
    values, the same points in every run."""
    from types import SimpleNamespace

    import numpy as np
    import torch

    sys.path.insert(0, str(ROOT))
    import bench

    g = torch.Generator().manual_seed(1)
    pred = SimpleNamespace(surf_vars={"2t": torch.randn(1, 1, 30, 40, generator=g)},
                           static_vars={"z": torch.randn(30, 40, generator=g)},
                           atmos_vars={"t": torch.randn(1, 1, 13, 30, 40, generator=g)})
    bench.dump_outputs(pred, tmp_path / "whole")
    assert sorted(f.name for f in (tmp_path / "whole").iterdir()) == ["atmos_t.npy", "static_z.npy", "surf_2t.npy"]
    assert np.array_equal(np.load(tmp_path / "whole" / "atmos_t.npy"), pred.atmos_vars["t"].numpy())
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 40_000)
    for run in ("a", "b"):
        bench.dump_outputs(pred, tmp_path / run)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 40_000
    for f in (tmp_path / "a").iterdir():
        sample = np.load(f)
        assert sample.dtype == np.float32 and sample.size > 0 and np.array_equal(sample, np.load(tmp_path / "b" / f.name))
        assert np.isin(sample, np.load(tmp_path / "whole" / f.name)).all()
