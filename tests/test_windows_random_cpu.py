"""Window / shift / mask index arithmetic on RANDOM geometries (no GPU): the C library's `__host__ __device__`
routine (the one the attention kernels use) against the oracle's closed form, structural invariants, and against the
reference's own roll -> pad -> window_partition_3d and compute_3d_shifted_window_mask on 120 further geometries (stored
as SHA-256 digests in tests/golden/windows_random.json, written by make_golden.py).  Extends the 34 stored golden
geometries to a few hundred."""

import json
from pathlib import Path

import numpy as np
import pytest
import torch

from aurora_b200 import cabi
from oracle import windows as W
from tests import fixtures as fx

WS0 = (2, 6, 12)
GOLD = Path(__file__).parent / "golden"
REFERENCE_CHUNKS = 4


def _geometries(n, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for _ in range(n):
        res = (int(rng.integers(1, 7)), int(rng.integers(1, 41)), int(rng.integers(1, 61)))
        out.append((res, bool(rng.integers(0, 2)), bool(rng.integers(0, 2))))
    return out


@pytest.mark.parametrize("chunk", range(6))
def test_host_map_equals_oracle_and_is_a_permutation(chunk):
    for res, shifted, warped in _geometries(40, 100 + chunk):
        ss0 = tuple(s // 2 for s in WS0) if shifted else (0, 0, 0)
        idx_o, ws, ss, nwin = W.window_gather_map(res, WS0, ss0)
        grp_o = W.window_group_ids(res, WS0, ss0, warped)
        idx_c, grp_c = cabi.window_index_map_host(res, WS0, ss0, warped)
        assert idx_c.shape == idx_o.shape, (res, shifted)
        np.testing.assert_array_equal(idx_c, idx_o.astype(np.int32), err_msg=str((res, shifted, warped)))
        if grp_o is not None:
            np.testing.assert_array_equal(grp_c, grp_o, err_msg=str((res, shifted, warped)))
        # every real token exactly once, the rest is padding
        real = idx_c[idx_c >= 0]
        n_tok = res[0] * res[1] * res[2]
        assert real.size == n_tok and np.array_equal(np.sort(real), np.arange(n_tok)), (res, shifted)
        assert (idx_c < 0).sum() == idx_c.size - n_tok
        if grp_o is not None:
            assert (grp_c[idx_c < 0] == W.PAD_GROUP).all() and (grp_c[idx_c >= 0] < W.PAD_GROUP).all()
        assert cabi.window_geometry(res, WS0, ss0)[:2] == idx_o.shape


@pytest.mark.parametrize("chunk", range(REFERENCE_CHUNKS))
def test_host_map_equals_reference_live(chunk):
    recs = json.loads((GOLD / "windows_random.json").read_text())[str(chunk)]
    assert [(tuple(r["res"]), r["shifted"], r["warped"]) for r in recs] == _geometries(30, 200 + chunk)
    compared = 0
    for rec in recs:
        res, shifted, warped = tuple(rec["res"]), rec["shifted"], rec["warped"]
        ss0 = tuple(s // 2 for s in WS0) if shifted else (0, 0, 0)
        idx_c, grp_c = cabi.window_index_map_host(res, WS0, ss0, warped)
        assert fx.array_digest(idx_c) == rec["idx"], (res, shifted)
        if rec["shift_after_adjust"]:
            if rec["mask"] is None:  # the reference's own `.view` fails on some degenerate grids (swin3d.py:355)
                continue
            assert fx.array_digest(grp_c) == rec["grp"], (res, shifted, warped)
            same = torch.from_numpy(grp_c)[:, :, None] == torch.from_numpy(grp_c)[:, None, :]
            assert fx.array_digest(torch.where(same, 0.0, -100.0)) == rec["mask"], (res, warped)
        compared += 1
    assert compared >= 20
