"""Rectification warp (SURVEY.md row a13) against the reference's own resampler.

The checker is oracle/_ref/homography_ref: the UNMODIFIED LibHomography / LibImages sources of the reference
compiled in place behind oracle/homography_harness.cpp.  The reference is float32 + SSE and is built with
-O3 -march=native, so its own output depends on FMA contraction: two builds of the same sources
(oracle/_ref/homography_ref vs homography_ref_nofma) differ by up to 6e-5 of the dynamic range on these inputs.
The tolerance below is set from that spread: |ours - reference| <= 1e-4 * max|src|, and the NaN (outside-the-source)
masks are identical except for pixels lying exactly on the source boundary.  The reference's outputs are stored by
tests/golden/reference_runs.py: the NaN mask in full, the values on a seeded sample of 2048 pixels."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_runs as RR  # noqa: E402

pytestmark = pytest.mark.gpu
REL_TOL = 1e-4


def _src(h=300, w=400, seed=0, nan=True):
    from s2p_b200.synth import _blur
    rng = np.random.default_rng(seed)
    a = _blur(rng.integers(0, 4096, size=(h, w)).astype(np.float64)).astype(np.float32)
    if nan:
        a[:20, :30] = np.nan
    return a


def _rot(th, s, tx, ty):
    c, si = np.cos(th) * s, np.sin(th) * s
    return np.array([[c, -si, tx], [si, c, ty], [0, 0, 1.0]])


CASES = {
    "identity": np.eye(3),
    "rot10": _rot(0.17, 1.0, 30, -40),
    "rot78_shrink": _rot(1.36, 0.9885, 250, -60),          # the fixtures' H_sec: min singular value 0.9885 -> AA branch
    "zoom_out": _rot(0.05, 0.6, 5, 5),
    "zoom_in": _rot(-0.1, 1.7, -60, 20),
    "perspective": np.array([[1.02, 0.03, -10], [0.01, 0.97, 5], [1e-5, -2e-5, 1]]),
    "shifted_crop": _rot(0.02, 1.0, -150, -100),           # needed ROI is a strict sub-window of the source
}


def warp_reference(oracle, name):
    """-> the stored reference resampler's output (reference_runs.Sample) for CASES[name] on _src(), 256 x 200"""
    return RR.reference_samples("warp/" + name, lambda: {"out": oracle.run_ref_homography(_src(), CASES[name], 256, 200)})["out"]


def dropin_reference(oracle):
    """-> (source, homography, stored reference output 200 x 150) of the file drop-in test"""
    src, H = _src(260, 340, seed=3, nan=False), _rot(0.12, 1.0, 20, -15)
    return src, H, RR.reference_samples("warp_dropin", lambda: {"out": oracle.run_ref_homography(src, H, 200, 150)})["out"]


def _assert_close(got, want, src, max_nan_diff):
    assert got.shape == want.shape
    nan_diff = int((want.isnan != np.isnan(got)).sum())
    assert nan_diff <= max_nan_diff, "%d NaN-mask mismatches" % nan_diff
    assert (~want.isnan & np.isfinite(got)).any()
    g = want.at(got)
    both = np.isfinite(want.val) & np.isfinite(g)
    err = np.abs(want.val[both] - g[both]).max()
    assert err <= REL_TOL * np.nanmax(np.abs(src)), "max abs error %g" % err


@pytest.mark.parametrize("name", sorted(CASES))
def test_warp_matches_reference(engine, oracle, name):
    want = warp_reference(oracle, name)
    got = engine.homography(_src(), CASES[name], 256, 200)
    assert got.shape == (200, 256)
    _assert_close(got, want, _src(), max(2, got.size // 5000))


def test_dropin_file_contract(engine, oracle, tmp_path):
    import subprocess
    from s2p_b200 import common, rasterio_compat as rio
    src, H, want = dropin_reference(oracle)
    im, out = str(tmp_path / "im.tif"), str(tmp_path / "rect.tif")
    rio.write_float_tiff(im, src)
    assert common.image_apply_homography(out, im, H, 200, 150) is None
    got = rio.read_band(out)
    assert got.shape == (150, 200)
    _assert_close(got, want, src, 2)
    with pytest.raises(subprocess.CalledProcessError):      # the binary exits with "empty roi"
        common.image_apply_homography(out, im, _rot(0, 1.0, 5000, 5000), 50, 50)


def test_dropin_warps_every_band(engine, oracle, tmp_path):
    """s2p/__init__.py:276 sends the multi-band colour image through image_apply_homography; the reference binary warps
    every band (3rdparty/homography/main.cpp loops over GetRasterCount)."""
    from s2p_b200 import common, rasterio_compat as rio
    bands = [_src(200, 260, seed=10 + k, nan=False) for k in range(3)]
    im, out = str(tmp_path / "clr.tif"), str(tmp_path / "clr_rect.tif")
    rio.write_float_tiff_bands(im, bands)
    H = _rot(-0.08, 1.0, 12, 9)
    common.image_apply_homography(out, im, H, 180, 140)
    assert rio.band_count(out) == 3
    for k in range(3):
        got = rio.read_window(out, 0, 0, 180, 140, k + 1)
        one = engine.homography(bands[k], H, 180, 140)
        assert np.array_equal(got, one, equal_nan=True)
    assert not np.array_equal(rio.read_window(out, 0, 0, 180, 140, 1), rio.read_window(out, 0, 0, 180, 140, 2), equal_nan=True)


def _real_pair():
    import make_golden_real_pair
    z = make_golden_real_pair.load()
    comp = lambda Hm, xy: np.asarray(Hm, np.float64) @ np.array([[1, 0, xy[0]], [0, 1, xy[1]], [0, 0, 1.0]])
    return z, comp(z["H1"], z["xy1"]), comp(z["H2"], z["xy2"])


def test_real_imagery_warp_golden(engine):
    """A golden the reference holds itself: tests/data/input_triangulation/pair_1/rectified_ref.tif is
    homography(img_01.tif, H_ref.txt) (fixture: tests/golden/make_golden_real_pair.py).  H is stored with 6 digits, which alone
    moves the result by 1.3e-4 of the range (measured with the reference resampler); tolerance 2e-4 of the range, NaN masks equal."""
    z, H1, _ = _real_pair()
    want = z["rectified_ref"]
    h, w = want.shape
    got = engine.homography(z["crop1"].astype(np.float32), H1, w, h)
    assert int((np.isnan(got) != np.isnan(want)).sum()) == 0
    both = np.isfinite(want)
    assert np.abs(got[both] - want[both]).max() <= 2e-4 * np.nanmax(want)


def test_real_imagery_chain_reproduces_reference_disparity(engine):
    """The whole hot path on real Pleiades imagery: warp img_02 with H_sec, match the reference's rectified_ref.tif against it
    on [-41, 30] (algo mgm) and compare with the disparity map the reference ships (rectified_disp.tif).  The reference's own
    `mgm` on the same rebuilt pair agrees with that map to <= 0.25 px on 99.72 % of the pixels (H_sec is stored with 6 digits
    and the shipped map predates the current matcher flags); the engine is held to >= 99.5 %."""
    from s2p_b200.engine import default_params
    z, _, H2 = _real_pair()
    ref, want = z["rectified_ref"], z["rectified_disp"]
    h, w = ref.shape
    sec = engine.homography(z["crop2"].astype(np.float32), H2, w, h)
    out = engine.mgm(ref, sec, -41, 30, default_params("mgm"))
    both = np.isfinite(out["disp"]) & np.isfinite(want)
    assert both.mean() > 0.9
    assert (np.abs(out["disp"][both] - want[both]) <= 0.25).mean() >= 0.995
    assert (np.isnan(out["disp"]) != np.isnan(want)).mean() < 0.01


def test_fused_rectify_and_match_equals_the_file_path(engine, tmp_path):
    """s2p_b200.fused.rectify_and_match (both warps and the matcher in one device call, the rectified pair never leaving the
    GPU) writes the same five files, bit for bit, as image_apply_homography x 2 followed by compute_disparity_map."""
    from s2p_b200 import block_matching as bm, common, fused, rasterio_compat as rio
    z, _, _ = _real_pair()
    a, b = str(tmp_path / "img_01.tif"), str(tmp_path / "img_02.tif")
    rio.write_float_tiff(a, z["crop1"].astype(np.float32))
    rio.write_float_tiff(b, z["crop2"].astype(np.float32))
    comp = lambda Hm, xy: np.asarray(Hm, np.float64) @ np.array([[1, 0, xy[0]], [0, 1, xy[1]], [0, 0, 1.0]])
    H1, H2 = comp(z["H1"], z["xy1"]), comp(z["H2"], z["xy2"])
    h, w = z["rectified_ref"].shape
    for algo in ("mgm", "mgm_multi"):
        d1 = tmp_path / ("two_step_" + algo)
        d2 = tmp_path / ("fused_" + algo)
        d1.mkdir(); d2.mkdir()
        p = lambda d, n: str(d / n)
        common.image_apply_homography(p(d1, "rectified_ref.tif"), a, H1, w, h)
        common.image_apply_homography(p(d1, "rectified_sec.tif"), b, H2, w, h)
        bm.compute_disparity_map(p(d1, "rectified_ref.tif"), p(d1, "rectified_sec.tif"), p(d1, "rectified_disp.tif"), p(d1, "rectified_mask.png"),
                                 algo, -41, 30)
        fused.rectify_and_match(p(d2, "rectified_ref.tif"), p(d2, "rectified_sec.tif"), p(d2, "rectified_disp.tif"), p(d2, "rectified_mask.png"),
                                a, b, H1, H2, w, h, algo, -41, 30)
        for name in ("rectified_ref.tif", "rectified_sec.tif", "rectified_disp.tif", "rectified_disp_confidence.tif", "rectified_mask.png"):
            assert np.array_equal(rio.read_band(p(d1, name)), rio.read_band(p(d2, name)), equal_nan=True), (algo, name)


def test_rectify_pair_and_match_with_the_reference_host_algebra(engine, tmp_path, monkeypatch):
    """rectification.rectify_pair_and_match lets the reference's rectify_pair do its host algebra, intercepts its two
    image_apply_homography calls and runs warps + matcher in one device call.  s2p is not importable here (rasterio, rpcm), so a
    stand-in module with rectify_pair's contract -- compute H1, H2, the range, then call common.image_apply_homography twice,
    s2p/rectification.py:367-382 -- takes its place; the files must equal those of the two-step drop-ins."""
    import sys
    import types
    from s2p_b200 import block_matching as bm, common, rasterio_compat as rio, rectification
    z, _, _ = _real_pair()
    a, b = str(tmp_path / "img_01.tif"), str(tmp_path / "img_02.tif")
    rio.write_float_tiff(a, z["crop1"].astype(np.float32))
    rio.write_float_tiff(b, z["crop2"].astype(np.float32))
    comp = lambda Hm, xy: np.asarray(Hm, np.float64) @ np.array([[1, 0, xy[0]], [0, 1, xy[1]], [0, 0, 1.0]])
    H1, H2 = comp(z["H1"], z["xy1"]), comp(z["H2"], z["xy2"])
    h, w = z["rectified_ref"].shape
    fake_common = types.ModuleType("s2p.common")
    fake_common.image_apply_homography = common.image_apply_homography
    fake_rect = types.ModuleType("s2p.rectification")

    def rectify_pair(im1, im2, rpc1, rpc2, x, y, ww, hh, out1, out2, A=None, sift_matches=None, method="rpc", hmargin=0, vmargin=0):
        fake_common.image_apply_homography(out1, im1, H1, w, h)
        fake_common.image_apply_homography(out2, im2, H2, w, h)
        return H1, H2, -41.0, 30.0
    fake_rect.rectify_pair = rectify_pair
    pkg = types.ModuleType("s2p")
    pkg.common, pkg.rectification = fake_common, fake_rect
    for name, mod in (("s2p", pkg), ("s2p.common", fake_common), ("s2p.rectification", fake_rect)):
        monkeypatch.setitem(sys.modules, name, mod)
    d1, d2 = tmp_path / "two_step", tmp_path / "fused"
    d1.mkdir(); d2.mkdir()
    p = lambda d, n: str(d / n)
    rectify_pair(a, b, None, None, 0, 0, w, h, p(d1, "rectified_ref.tif"), p(d1, "rectified_sec.tif"))
    bm.compute_disparity_map(p(d1, "rectified_ref.tif"), p(d1, "rectified_sec.tif"), p(d1, "rectified_disp.tif"), p(d1, "rectified_mask.png"), "mgm", -41.0, 30.0)
    ret = rectification.rectify_pair_and_match(a, b, None, None, 0, 0, w, h, p(d2, "rectified_ref.tif"), p(d2, "rectified_sec.tif"),
                                               p(d2, "rectified_disp.tif"), p(d2, "rectified_mask.png"), "mgm")
    assert ret[2:] == (-41.0, 30.0) and fake_common.image_apply_homography is common.image_apply_homography      # patch restored
    for name in ("rectified_ref.tif", "rectified_sec.tif", "rectified_disp.tif", "rectified_disp_confidence.tif", "rectified_mask.png"):
        assert np.array_equal(rio.read_band(p(d1, name)), rio.read_band(p(d2, name)), equal_nan=True), name
