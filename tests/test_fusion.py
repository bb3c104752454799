"""n-view merge (SURVEY.md section 8f rank 1): the numpy restatement against the stored results of the reference's own
`average_if_close` (CPU), and the CUDA kernel against the restatement (GPU).  Bit-exact."""
import os
import sys

import numpy as np
import pytest

from util import same

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_runs as RR  # noqa: E402


def _maps(n, h=37, w=53, seed=0):
    rng = np.random.default_rng(seed)
    base = rng.normal(100, 5, (h, w))
    maps = [(base + rng.normal(0, 0.7, (h, w)) + 3 * k).astype(np.float32) for k in range(n)]
    for m in maps:
        m[rng.random((h, w)) < 0.25] = np.nan
    maps[0][:3] = np.nan
    for m in maps:
        m[5, :7] = np.nan                     # an all-NaN run
    offsets = [3.0 * k + 0.1234567 for k in range(n)]
    return maps, offsets


@pytest.mark.parametrize("n", [2, 3, 5])
def test_port_matches_reference_function(n):
    from oracle import fusion_oracle as F
    maps, offsets = _maps(n, seed=n)
    for thr in (1, 3):
        want = RR.reference_digests("average_if_close/n=%d,threshold=%d" % (n, thr), lambda: {"merged": F.merge_ref(maps, offsets, thr)})
        bad = RR.mismatches({"merged": F.merge_port(maps, offsets, "average_if_close", thr)}, want)
        assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("n,op", [(2, "average_if_close"), (3, "average_if_close"), (4, "np.nanmedian"), (3, "np.nanmean"),
                                  (5, "np.nanmin"), (2, "np.nanmax"), (3, "np.median"), (4, "np.mean"), (2, "np.min"), (3, "np.max"),
                                  (9, "np.nanmean"), (13, "np.mean"), (16, "np.nanmean")])
@pytest.mark.parametrize("sub_f32", [None, True, False])
def test_gpu_merge_matches_port(engine, n, op, sub_f32):
    """sub_f32: the offsets are subtracted in float32 (NumPy < 2) or float64 (NumPy >= 2); None = whatever the NumPy of
    this environment does with the reference's own expression.  n >= 8 exercises NumPy's pairwise summation."""
    from oracle import fusion_oracle as F
    maps, offsets = _maps(n, seed=10 + n)
    if op in ("np.mean", "np.median", "np.min", "np.max"):
        for m in maps[1:]:
            m[np.isnan(m) & (np.arange(m.shape[1])[None, :] % 3 > 0)] = 101.5     # leave pixels where no value is NaN
    got = engine.merge_n(maps, offsets, op, threshold=3, sub_f32=sub_f32)
    want = F.merge_port(maps, offsets, op, 3, sub_f32=sub_f32)
    assert same(got, want), "%d px differ" % int((~((got == want) | (np.isnan(got) & np.isnan(want)))).sum())


@pytest.mark.gpu
def test_gpu_merge_dropin_files(engine, tmp_path):
    from oracle import fusion_oracle as F
    from s2p_b200 import fusion, rasterio_compat as rio
    maps, offsets = _maps(2, seed=77)
    paths = []
    for k, m in enumerate(maps):
        p = str(tmp_path / ("height_map_%d.tif" % k))
        rio.write_float_tiff(p, m)
        paths.append(p)
    out = str(tmp_path / "height_map.tif")
    fusion.merge_n(out, paths, offsets, averaging="average_if_close", threshold=3)
    assert same(rio.read_band(out), F.merge_port(maps, offsets, "average_if_close", 3))


EROSION_RADII = [2, 3, 5]


def erosion_reference(oracle, radius):
    """-> (mask, stored digests of the reference's erosion of it)"""
    rng = np.random.default_rng(radius)
    m = (rng.random((61, 83)) > 0.15).astype(np.uint8)
    want = RR.reference_digests("disk_erosion/%d" % radius,
                                lambda: {"mask": oracle.ref_disk_erosion(m.astype(np.float32), radius).astype(np.uint8)})
    return m, want


@pytest.mark.gpu
@pytest.mark.parametrize("radius", EROSION_RADII)
def test_gpu_mask_erosion_matches_reference(engine, oracle, radius, tmp_path):
    """masking.erosion = `morsi diskR erosion` (c/morsi.c compiled in place as oracle/_ref/libmorsi_ref.so; its results are
    stored by tests/golden/reference_runs.py)."""
    m, want = erosion_reference(oracle, radius)
    assert not RR.mismatches({"mask": engine.erode_mask(m, radius)}, want)
    if radius == 2:       # file-level drop-in (s2p/masking.py:87-97)
        from s2p_b200 import masking, rasterio_compat as rio
        p = str(tmp_path / "rectified_mask.png")
        rio.write_mask_png(p, m)
        masking.erosion(p, p, 2)
        assert not RR.mismatches({"mask": rio.read_band(p).astype(np.uint8)}, want)
        rio.write_mask_png(p, m)
        masking.erosion(p, p, 1)                      # below 2: untouched, as in the reference
        assert np.array_equal(rio.read_band(p).astype(np.uint8), m)
