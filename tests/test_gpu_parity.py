"""GPU parity proper: the CUDA path (through the C ABI) against the CPU oracle on the same
seeded inputs.  Bit-exact for the integer WTA index, confidence, mask and -- because the
device arithmetic follows the reference's float32 operation order -- for the sub-pixel map too
(the contract only asks +-0.25 px; both are asserted, the tolerance stated here)."""
import os
import sys

import numpy as np
import pytest

from s2p_b200.synth import make_pair
from util import nmismatch, same

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_runs as RR  # noqa: E402

pytestmark = pytest.mark.gpu
SUBPIX_TOL = 0.25  # px, BASELINE.json north_star


def _ranges(h, w, dmin, dmax):
    return np.full((h, w), dmin, np.int32), np.full((h, w), dmax, np.int32)


@pytest.mark.parametrize("win", [5, 3, 7])
def test_census(engine, oracle, win):
    ref, _, _ = make_pair(61, 83, -8, 8, seed=11)
    assert np.array_equal(engine.census(ref, win), oracle.port.census(ref, win))


@pytest.mark.parametrize("win,dmin,dmax", [(5, -12, 11), (3, -5, 20), (7, -40, 2), (5, -64, 63)])
def test_costvolume(engine, oracle, win, dmin, dmax):
    h, w = 37, 150
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=3)
    lo, hi = _ranges(h, w, dmin, dmax)
    lo[5:9, 10:40] = dmin + 1            # ragged per-pixel ranges
    hi[5:9, 10:40] = dmin + 3
    D = dmax - dmin + 1
    Cg = engine.costvolume(ref, sec, lo, hi, dmin, D, win)
    Co = oracle.port.costvolume(ref, sec, lo, hi, dmin, D, win)
    assert same(Cg, Co)


@pytest.mark.parametrize("tsgm", [1, 2, 3, 4])
@pytest.mark.parametrize("ndir", [8, 4])
def test_aggregate(engine, oracle, tsgm, ndir):
    h, w, dmin, dmax = 45, 70, -10, 13
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=5)
    lo, hi = _ranges(h, w, dmin, dmax)
    lo[20:24, 30:50] = dmin
    hi[20:24, 30:50] = dmin + 1
    D = dmax - dmin + 1
    C = oracle.port.costvolume(ref, sec, lo, hi, dmin, D, 5)
    So, do, co, fo = oracle.port.aggregate(C, lo, hi, dmin, 8.0, 32.0, ndir, tsgm)
    Sg, dg, cg, fg = engine.aggregate(C, lo, hi, dmin, 8.0, 32.0, ndir, tsgm)
    assert same(dg, do), "integer WTA index differs at %d pixels" % nmismatch(dg, do)
    assert same(fg, fo), "consensus differs at %d pixels" % nmismatch(fg, fo)
    assert same(Sg, So), "aggregated volume differs at %d voxels" % nmismatch(Sg, So)
    assert same(cg, co)


@pytest.mark.parametrize("shape,dmin,dmax,nanb,seed", [
    ((64, 96), -12, 11, 0.0, 1),      # D=24  -> 1 label per lane
    ((50, 81), -20, 30, 0.0, 2),      # D=51  -> 2
    ((40, 130), -64, 63, 0.0, 3),     # D=128 -> 4
    ((33, 140), -64, 63, 0.06, 4),    # no-data in both images: right hull sticks out -> 5
    ((30, 200), -90, 70, 0.0, 5),     # D=161 -> 6
    ((24, 260), -128, 127, 0.0, 6),   # D=256 -> 8
    ((70, 45), 3, 19, 0.05, 7),       # positive range, more rows than columns, no-data
    ((20, 400), -150, 150, 0.0, 8),   # D=301 -> 12
    ((18, 520), -250, 249, 0.03, 9),  # D=500 -> 16 (the widest slab)
])
def test_mgm_end_to_end(engine, oracle, shape, dmin, dmax, nanb, seed):
    h, w = shape
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=seed, nan_border=nanb)
    from s2p_b200.engine import default_params
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm"), want_mask=True, want_right=True)
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params())
    m = oracle.port.rejection_mask(d, ref, sec)
    both = np.isfinite(d) & np.isfinite(out["disp"])
    assert np.array_equal(np.isnan(d), np.isnan(out["disp"]))
    assert np.all(np.abs(d[both] - out["disp"][both]) <= SUBPIX_TOL)
    assert same(out["disp"], d), "sub-pixel disparity not bit-exact at %d px" % nmismatch(out["disp"], d)
    assert same(out["conf"], c), "confidence differs at %d px" % nmismatch(out["conf"], c)
    assert same(out["disp_right"], dr)
    assert np.array_equal(out["mask"], m)


@pytest.mark.parametrize("kw", [dict(tsgm=4), dict(tsgm=2), dict(ndir=4), dict(census_win=3), dict(census_win=7),
                                dict(median=0, lr_mode=0, refine=0), dict(median=2), dict(P1=4.0, P2=50.0), dict(mindiff=1.0),
                                dict(mindiff=0.5, median=0)])
def test_mgm_options(engine, oracle, kw):
    h, w, dmin, dmax = 48, 90, -9, 14
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=21, nan_border=0.04)
    from s2p_b200.engine import default_params
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm", **kw), want_right=True)
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params(**kw))
    assert same(out["disp"], d), "disparity differs at %d px" % nmismatch(out["disp"], d)
    assert same(out["conf"], c)
    assert same(out["disp_right"], dr)


def test_median_and_mask(engine, oracle):
    rng = np.random.default_rng(0)
    a = rng.normal(size=(40, 50)).astype(np.float32)
    a[rng.random(a.shape) < 0.2] = np.nan
    for r in (1, 2):
        assert same(engine.median(a, r), oracle.port.median(a, r))
    ref, sec, gt = make_pair(40, 50, -6, 6, seed=9, nan_border=0.1)
    d = gt + rng.uniform(-0.5, 0.5, gt.shape).astype(np.float32)
    d[rng.random(d.shape) < 0.1] = np.nan
    assert np.array_equal(engine.rejection_mask(d, ref, sec), oracle.port.rejection_mask(d, ref, sec))


def test_batch_matches_single(engine):
    from s2p_b200.engine import default_params
    h, w, dmin, dmax = 40, 64, -8, 7
    pairs = [make_pair(h, w, dmin, dmax, seed=s)[:2] for s in range(5)]
    engine.reserve(3, w, h, dmax - dmin + 1)
    p = default_params("mgm")
    disp, conf, mask = engine.mgm_batch([a for a, _ in pairs], [b for _, b in pairs], dmin, dmax, p)
    for k, (a, b) in enumerate(pairs):
        one = engine.mgm(a, b, dmin, dmax, p)
        assert same(disp[k], one["disp"]) and same(conf[k], one["conf"]) and np.array_equal(mask[k], one["mask"])


def test_timeout_and_errors(engine):
    from s2p_b200 import _lib
    from s2p_b200.engine import S2pbError, default_params
    ref, sec, _ = make_pair(512, 512, -100, 100, seed=1)
    with pytest.raises(S2pbError) as e:
        engine.mgm(ref, sec, -100, 100, default_params("mgm", timeout_ms=1))
    assert e.value.code == _lib.ERR_TIMEOUT
    # the context stays usable after an aborted call
    out = engine.mgm(ref[:64, :64], sec[:64, :64], -8, 8, default_params("mgm"))
    assert np.isfinite(out["disp"]).any()
    with pytest.raises(S2pbError) as e:
        engine.mgm(ref, sec, 5, 5, default_params("mgm"))
    assert e.value.code == _lib.ERR_ARG


@pytest.mark.parametrize("name", ["plain", "wide", "nan_ref", "nan_both", "tsgm4_o4", "census3", "multi", "multi_s1", "real", "real_multi"])
def test_against_reference_golden_vectors(engine, name):
    """tests/golden/*.npz are outputs of the unmodified reference binary (tests/golden/make_golden.py)."""
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    import make_golden as G
    from s2p_b200.engine import default_params
    ref, sec, dmin, dmax, kw = G.inputs(name)
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    algo, kw = G.split_kw(kw)
    out = engine.mgm(ref, sec, dmin, dmax, default_params(algo, **kw), want_right=True)
    assert same(out["disp"], g["disp"]), "%d px differ from the reference" % nmismatch(out["disp"], g["disp"])
    assert np.array_equal(out["conf"].astype(np.uint8), g["conf"])
    assert same(out["disp_right"], g["dispR"])


def test_dropin_file_contract(engine, oracle, tmp_path):
    """compute_disparity_map: same signature, files and exceptions as s2p/block_matching.py:35-336."""
    import subprocess
    from s2p_b200 import block_matching as bm, rasterio_compat as rio
    h, w, dmin, dmax = 60, 100, -11, 12
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=42, nan_border=0.05)
    im1, im2 = str(tmp_path / "rectified_ref.tif"), str(tmp_path / "rectified_sec.tif")
    disp, mask = str(tmp_path / "rectified_disp.tif"), str(tmp_path / "rectified_mask.png")
    rio.write_float_tiff(im1, ref)
    rio.write_float_tiff(im2, sec)
    assert bm.compute_disparity_map(im1, im2, disp, mask, "mgm", dmin + 0.4, dmax - 0.3) is None
    d, c, _ = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params())
    m = oracle.port.rejection_mask(d, ref, sec)
    assert same(rio.read_band(disp), d)
    assert same(rio.read_band(bm.confidence_path(disp)), c)
    assert np.array_equal(rio.read_band(mask).astype(np.uint8), m)
    with pytest.raises(bm.MaxDisparityRangeError):
        bm.compute_disparity_map(im1, im2, disp, mask, "mgm", -100, 100, max_disp_range=10)
    big_ref, big_sec, _ = make_pair(512, 512, -100, 100, seed=1)
    rio.write_float_tiff(im1, big_ref)
    rio.write_float_tiff(im2, big_sec)
    with pytest.raises(subprocess.TimeoutExpired):      # tests/block_matching_test.py:18-21 in the reference
        bm.compute_disparity_map(im1, im2, disp, mask, "mgm", -100, 100, timeout=0.001)


@pytest.mark.parametrize("shape,dmin,dmax,nanb,seed,kw", [
    ((120, 160), -20, 20, 0.0, 1, dict(subpix=1)),                 # pyramid only
    ((120, 160), -20, 20, 0.0, 1, dict()),                         # + half-pixel pass (SUBPIX=2)
    ((130, 210), -30, 25, 0.0, 2, dict()),
    ((230, 260), -40, 40, 0.0, 3, dict(scales=3)),
    ((110, 150), -12, 18, 0.0, 4, dict(lr_mode=2, remove_small_cc=0)),
    ((130, 170), -14, 16, 0.06, 5, dict()),                        # no-data strips in both images, every pyramid level
    ((120, 160), -20, 20, 0.05, 6, dict(subpix=1)),
])
def test_mgm_multi(engine, oracle, shape, dmin, dmax, nanb, seed, kw):
    """mgm_multi (s2p flags: -S 6, SUBPIX=2, REMOVESMALLCC=25, TSGM=4): bit-exact, including the half-pixel pass -- the
    engine evaluates the reference's DCT shift with the same tables and summation order (dct_kernels.cuh)."""
    from s2p_b200.engine import default_params
    h, w = shape
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=seed, nan_border=nanb)
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm_multi", **kw), want_right=True)
    d, c, dr = oracle.port.mgm_multi(ref, sec, dmin, dmax, oracle.mgm_multi_params(**kw))
    assert same(out["conf"], c), "consensus (ZOOM=1 call) differs at %d px" % nmismatch(out["conf"], c)
    assert same(out["disp"], d), "%d px differ" % nmismatch(out["disp"], d)
    assert same(out["disp_right"], dr)


@pytest.mark.parametrize("shape,dmin,dmax", [((2, 2), -1, 1), ((3, 9), -2, 3), ((9, 3), -4, 1), ((17, 5), 0, 6), ((6, 40), -20, 20),
                                             ((33, 34), -3, 2), ((150, 7), -5, 5)])
def test_tiny_and_thin_tiles(engine, oracle, shape, dmin, dmax):
    """Shapes smaller than a band (16 scanlines), than the cp.async pipeline (8 pixels) or than the census window."""
    from s2p_b200.engine import default_params
    h, w = shape
    rng = np.random.default_rng(h * 100 + w)
    ref = rng.integers(0, 4096, (h, w)).astype(np.float32)
    sec = np.roll(ref, 1, axis=1) + rng.normal(0, 20, (h, w)).astype(np.float32)
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm"), want_right=True)
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params())
    assert same(out["disp"], d) and same(out["conf"], c) and same(out["disp_right"], dr)
    assert np.array_equal(out["mask"], oracle.port.rejection_mask(d, ref, sec))


def test_mgm_multi_batch_and_file_dropin(engine, oracle, tmp_path):
    """algo='mgm_multi' through the batch entry point and through compute_disparity_map."""
    from s2p_b200 import block_matching as bm, rasterio_compat as rio
    from s2p_b200.engine import default_params
    h, w, dmin, dmax = 110, 130, -9, 12
    pairs = [make_pair(h, w, dmin, dmax, seed=60 + k)[:2] for k in range(3)]
    p = default_params("mgm_multi")
    disp, conf, mask = engine.mgm_batch([a for a, _ in pairs], [b for _, b in pairs], dmin, dmax, p)
    for k, (a, b) in enumerate(pairs):
        one = engine.mgm(a, b, dmin, dmax, p)
        assert same(disp[k], one["disp"]) and same(conf[k], one["conf"]) and np.array_equal(mask[k], one["mask"])
    im1, im2 = str(tmp_path / "a.tif"), str(tmp_path / "b.tif")
    dpath, mpath = str(tmp_path / "d.tif"), str(tmp_path / "m.png")
    rio.write_float_tiff(im1, pairs[0][0])
    rio.write_float_tiff(im2, pairs[0][1])
    bm.compute_disparity_map(im1, im2, dpath, mpath, "mgm_multi", dmin, dmax)
    assert same(rio.read_band(dpath), disp[0])
    assert same(rio.read_band(bm.confidence_path(dpath)), conf[0])


@pytest.mark.gpu
def test_batch_page_locked_buffers_match_staged(engine):
    """Page-locked caller buffers are DMA'd directly (no staging copy); results must equal the staged path."""
    import torch
    from s2p_b200.engine import default_params
    eng = engine
    p = default_params("mgm")
    pairs = [make_pair(70, 96, -12, 9, seed=40 + k, nan_border=0.05 if k == 1 else 0.0) for k in range(3)]
    refs = [r for r, _, _ in pairs]
    secs = [s for _, s, _ in pairs]
    d0, c0, m0 = eng.mgm_batch(refs, secs, -12, 9, p)
    keep = []

    def pin(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
        keep.append(t)
        return t.numpy()
    outs = ([pin(np.zeros((70, 96), np.float32)) for _ in pairs], [pin(np.zeros((70, 96), np.float32)) for _ in pairs],
            [pin(np.zeros((70, 96), np.uint8)) for _ in pairs])
    d1, c1, m1 = eng.mgm_batch([pin(r) for r in refs], [pin(s) for s in secs], -12, 9, p, out=outs)
    for k in range(3):
        np.testing.assert_array_equal(d0[k], d1[k])
        np.testing.assert_array_equal(c0[k], c1[k])
        np.testing.assert_array_equal(m0[k], m1[k])
    with pytest.raises(ValueError):
        eng.mgm_batch(refs, secs, -12, 9, p, out=(outs[0][:2], outs[1], outs[2]))


NODATA_CASES = [((56, 88), -10, 9, 0.07, 106), ((90, 203), -24, 23, 0.05, 7), ((64, 333), -9, 40, 0.1, 8)]


def nodata_reference(oracle, shape, dmin, dmax, nanb, seed):
    """-> (ref, sec, stored digests of the reference binary's disp / conf / dispR on them)"""
    h, w = shape
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=seed, nan_border=nanb)

    def run():
        r = oracle.run_ref(ref, sec, dmin, dmax, oracle.mgm_params(), threads=1)
        return {k: r[k] for k in ("disp", "conf", "dispR")}
    return ref, sec, RR.reference_digests("nodata/%dx%d,seed=%d" % (h, w, seed), run)


@pytest.mark.parametrize("shape,dmin,dmax,nanb,seed", NODATA_CASES)
def test_nodata_matches_reference_binary(engine, oracle, shape, dmin, dmax, nanb, seed):
    """No-data in BOTH images: the reference's DCT round trip of the matched image leaves rounding noise on the zeroed
    pixels (mgm_costvolume.cc:23-60), which the census transform then compares.  The engine reproduces the round trip with
    the same tables and summation order, so it equals the unmodified reference binary bit for bit on such tiles too
    (its outputs are stored by tests/golden/reference_runs.py)."""
    from s2p_b200.engine import default_params
    ref, sec, want = nodata_reference(oracle, shape, dmin, dmax, nanb, seed)
    assert np.isnan(ref).any() and np.isnan(sec).any()
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm"), want_right=True)
    bad = RR.mismatches(dict(disp=out["disp"], conf=out["conf"], dispR=out["disp_right"]), want)
    assert not bad, "differs from the reference binary: " + "; ".join(bad)


def test_exact_zero_pixels_without_nodata(engine, oracle):
    """Pixels that are exactly 0 (or tiny against their row) without being no-data take the same path."""
    from s2p_b200.engine import default_params
    rng = np.random.default_rng(5)
    h, w, dmin, dmax = 50, 120, -9, 8
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=77)
    for im in (ref, sec):
        im[rng.random(im.shape) < 0.08] = 0.0
        im[rng.random(im.shape) < 0.02] = 1e-3
        im[10:14] = 0.0                       # whole rows of zeros come back as exact zeros
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm"), want_right=True)
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params())
    assert same(out["disp"], d) and same(out["conf"], c) and same(out["disp_right"], dr)


@pytest.mark.parametrize("name", ["c2_plain", "c2_nodata"])
def test_full_size_tile_matches_reference_binary(engine, name):
    """BASELINE configs[1] at its full size: one 1024 x 1024 x 128 tile against the digests of the unmodified reference
    binary's output (tests/golden/full_c2.json, generator tests/golden/make_golden_full.py), block of 32 rows by block."""
    import json
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from make_golden_full import digests
    from s2p_b200.engine import default_params
    path = os.path.join(os.path.dirname(__file__), "golden", "full_c2.json")
    if not os.path.exists(path):
        pytest.skip("tests/golden/full_c2.json not generated")
    g = json.load(open(path))[name]
    ref, sec, _ = make_pair(g["h"], g["w"], g["dmin"], g["dmax"], seed=g["seed"], nan_border=g["nan_border"])
    out = engine.mgm(ref, sec, g["dmin"], g["dmax"], default_params("mgm"), want_right=True)
    for key, arr in (("disp", out["disp"]), ("conf", out["conf"]), ("dispR", out["disp_right"])):
        got = digests(arr)
        bad = [k for k, (a, b) in enumerate(zip(got, g[key])) if a != b]
        assert not bad, "%s differs from the reference binary in %d of %d row blocks (first: rows %d..)" % (
            key, len(bad), len(got), bad[0] * g["block_rows"])


def test_eight_tiles_in_flight_equal_serial(engine):
    """What bench.py times: >= 8 DISTINCT tiles through s2pb_mgm_batch with 8 workspaces in flight (the WTA of one tile
    overlaps the aggregation of the next, copies overlap both), each compared with its own serial result."""
    from s2p_b200.engine import default_params
    h, w, dmin, dmax = 200, 320, -40, 39
    pairs = [make_pair(h, w, dmin, dmax, seed=300 + k, nan_border=0.04 if k % 3 == 1 else 0.0)[:2] for k in range(11)]
    p = default_params("mgm")
    serial = [engine.mgm(a, b, dmin, dmax, p) for a, b in pairs]
    engine.reserve(8, w, h, dmax - dmin + 2)
    for _ in range(2):          # the second pass reuses warm workspaces
        disp, conf, mask = engine.mgm_batch([a for a, _ in pairs], [b for _, b in pairs], dmin, dmax, p)
        for k, one in enumerate(serial):
            assert same(disp[k], one["disp"]), "tile %d: %d px differ" % (k, nmismatch(disp[k], one["disp"]))
            assert same(conf[k], one["conf"]) and np.array_equal(mask[k], one["mask"])


def rejection_mask_reference(oracle):
    """-> [(disp, ref, sec, stored digests of the reference programs' mask)] for two tiles"""
    rng = np.random.default_rng(4)
    out = []
    for seed, (h, w, dmin, dmax) in enumerate([(70, 110, -12, 12), (45, 200, -30, 8)]):
        ref, sec, gt = make_pair(h, w, dmin, dmax, seed=50 + seed, nan_border=0.06)
        d = gt + rng.uniform(-0.7, 0.7, gt.shape).astype(np.float32)
        d[rng.random(d.shape) < 0.1] = np.nan
        d[:, :3] -= 7.3
        want = RR.reference_digests("rejection_mask_gpu/%d" % seed, lambda: {"mask": oracle.ref_rejection_mask(d, ref, sec)})
        out.append((d, ref, sec, want))
    return out


def test_rejection_mask_matches_reference_programs(engine, oracle):
    """the mask kernel against the reference's own plambda / backflow / plambda chain (oracle/_ref, c/*.c compiled in place; its
    results are stored by tests/golden/reference_runs.py)"""
    for d, ref, sec, want in rejection_mask_reference(oracle):
        bad = RR.mismatches({"mask": engine.rejection_mask(d, ref, sec)}, want)
        assert not bad, bad


def test_mgm_multi_level_hull_wider_than_512_labels(engine, oracle):
    """A pyramid level whose label hull exceeds 512 labels (here the half-pixel pass of a 190-label range with the no-data
    sentinel sticking out): the reference has no such limit (mgm_costvolume.cc:63-72, one vector per pixel); the engine
    serves it through the chunk-skipping kernels."""
    from s2p_b200.engine import default_params
    h, w, dmin, dmax = 123, 191, -128, 61
    kw = dict(ndir=2, tsgm=4, census_win=3, P1=8.0, P2=48.0, median=1, lr_mode=0)
    for seed, nanb in ((5, 0.05), (6, 0.0)):
        ref, sec, _ = make_pair(h, w, dmin, dmax, seed=seed, nan_border=nanb)
        out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm_multi", **kw), want_right=True)
        d, c, dr = oracle.port.mgm_multi(ref, sec, dmin, dmax, oracle.mgm_multi_params(**kw))
        assert same(out["disp"], d), "%d px differ" % nmismatch(out["disp"], d)
        assert same(out["conf"], c) and same(out["disp_right"], dr)


@pytest.mark.parametrize("dmin,dmax,tsgm", [(-300, 299, 3), (-20, 560, 4), (-700, 450, 2)])
def test_mgm_more_than_512_labels(engine, oracle, dmin, dmax, tsgm):
    """algo mgm with a disparity range beyond the 512 labels of the register-resident kernels (up to 2048 are served)"""
    from s2p_b200.engine import default_params
    h, w = 37, 640
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=dmax, nan_border=0.03)
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm", tsgm=tsgm), want_right=True)
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params(tsgm=tsgm))
    assert same(out["disp"], d), "%d px differ" % nmismatch(out["disp"], d)
    assert same(out["conf"], c) and same(out["disp_right"], dr)


@pytest.mark.parametrize("algo,shape,dmin,dmax,nanb,kw", [
    ("mgm", (70, 110), -12, 12, 0.05, {}), ("mgm", (45, 200), -30, 8, 0.0, dict(tsgm=4, census_win=3)), ("mgm", (37, 640), -300, 299, 0.03, {}),
    ("mgm_multi", (120, 160), -20, 20, 0.0, {}), ("mgm_multi", (130, 170), -14, 16, 0.06, dict(subpix=1))])
def test_pkr_confidence(engine, oracle, algo, shape, dmin, dmax, nanb, kw):
    """the peak-ratio confidence images of -confidence_pkrL / -confidence_pkrR (mgm_costvolume.cc:199-214), bit for bit; the oracle
    is pinned to the reference binary's own images (tests/test_oracle.py)"""
    from s2p_b200.engine import default_params
    h, w = shape
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=h + w, nan_border=nanb)
    multi = algo == "mgm_multi"
    out = engine.mgm(ref, sec, dmin, dmax, default_params(algo, **kw), want_right=True, want_pkr=True)
    P = oracle.mgm_multi_params(**kw) if multi else oracle.mgm_params(**kw)
    d, c, dr, pl, pr = oracle.port.mgm_pkr(ref, sec, dmin, dmax, P, multi=multi)
    assert same(out["disp"], d) and same(out["conf"], c) and same(out["disp_right"], dr)
    assert same(out["pkr_left"], pl), "%d px differ" % nmismatch(out["pkr_left"], pl)
    assert same(out["pkr_right"], pr), "%d px differ" % nmismatch(out["pkr_right"], pr)


def test_nodata_with_a_ragged_mask(engine, oracle):
    """No-data regions as a real rectified tile has them: a rotated footprint, so that every row loses another set of columns (the
    column list of the inverse DCT grows to most of the width), plus isolated exact zeros."""
    from s2p_b200.engine import default_params
    h, w, dmin, dmax = 96, 180, -14, 13
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=21)
    yy, xx = np.mgrid[0:h, 0:w]
    ref[xx + 2 * yy < 60] = np.nan
    ref[xx - yy > 150] = np.nan
    sec[3 * xx + yy < 70] = np.nan
    sec[xx + yy > 230] = np.nan
    sec[40:44, 90:95] = 0.0
    out = engine.mgm(ref, sec, dmin, dmax, default_params("mgm"), want_right=True)
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params())
    assert same(out["disp"], d), "%d px differ" % nmismatch(out["disp"], d)
    assert same(out["conf"], c) and same(out["disp_right"], dr)
