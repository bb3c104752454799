"""Triangulation (SURVEY.md section 8f rank 2): the CUDA kernel against the reference's own disp_to_lonlatalt
(c/disp_to_h.c + c/rpc.c compiled in place as oracle/_ref/libdisp_to_h_ref.so).  float64 iterative geometry built
-O3 -march=native on the reference side: tolerance 1e-9 degree (~0.1 mm) on lon/lat, 1e-6 m on the altitude,
1e-4 px on the reprojection error, identical NaN pattern.  The reference library's outputs are stored by
tests/golden/reference_runs.py: the NaN patterns in full, the values on a seeded sample of pixels."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import reference_runs as RR  # noqa: E402

pytestmark = pytest.mark.gpu


def _rpc(seed, with_direct):
    """A synthetic but geometrically consistent camera: affine ground->image model with a mild cubic ripple."""
    from s2p_b200.triangulation import RPCStruct
    rng = np.random.default_rng(seed)
    r = RPCStruct()
    for k in range(20):
        r.inumx[k] = r.idenx[k] = r.inumy[k] = r.ideny[k] = 0.0
        r.numx[k] = r.denx[k] = r.numy[k] = r.deny[k] = np.nan
    r.idenx[0] = r.ideny[0] = 1.0
    # normalised col = f(lon, lat, alt): polynomial variables of c/rpc.c:279-297 are (1, lat?, ...) with the x/y swap
    a = 0.9 + 0.05 * rng.random(); b = 0.1 * (rng.random() - 0.5); c = 0.35 * (rng.random() - 0.3)
    r.inumx[1], r.inumx[2], r.inumx[3] = b, a, c          # col ~ a*lon + b*lat + c*alt
    r.inumy[1], r.inumy[2], r.inumy[3] = -a, b * 0.5, 0.02  # row ~ -a*lat + ...
    r.inumx[4] = 1e-3; r.inumy[7] = -2e-3; r.idenx[3] = 1e-3; r.ideny[1] = 5e-4
    r.scale[0], r.scale[1], r.scale[2] = 5000.0, 4000.0, 500.0
    r.offset[0], r.offset[1], r.offset[2] = 5000.0, 4000.0, 100.0
    r.iscale[0], r.iscale[1], r.iscale[2] = 0.05, 0.04, 500.0
    r.ioffset[0], r.ioffset[1], r.ioffset[2] = 2.3, 48.8, 100.0
    r.delta = 1.0
    if with_direct:       # a crude direct model (exact inverse of the linear part): exercises the non-iterative branch
        for k in range(20):
            r.numx[k] = r.denx[k] = r.numy[k] = r.deny[k] = 0.0
        r.denx[0] = r.deny[0] = 1.0
        M = np.array([[a, b], [b * 0.5, -a]])
        Mi = np.linalg.inv(M)
        r.numx[2], r.numx[1], r.numx[3] = Mi[0, 0], Mi[0, 1], -(Mi[0, 0] * c + Mi[0, 1] * 0.02)
        r.numy[2], r.numy[1], r.numy[3] = Mi[1, 0], Mi[1, 1], -(Mi[1, 0] * c + Mi[1, 1] * 0.02)
    return r


def _geometry():
    """Rectifying homographies that send the image window around (4200, 3290) to the rectified tile's origin."""
    def hom(A, origin, persp=0.0):
        A = np.asarray(A, float)
        t = -A @ np.asarray(origin, float)
        return np.array([[A[0, 0], A[0, 1], t[0]], [A[1, 0], A[1, 1], t[1]], [persp, 0, 1.0]])
    H1 = hom([[0.99, 0.05], [-0.04, 1.01]], (4200.0, 3290.0))
    H2 = hom([[1.0, 0.03], [-0.02, 0.99]], (4195.0, 3288.0), 1e-7)
    return H1, H2, (4180.0, 4330.0, 3280.0, 3390.0)


def _assert_matches(got, gerr, want, min_valid):
    w, werr = want["lonlatalt"], want["err"]
    assert np.array_equal(w.isnan, np.isnan(got)) and np.array_equal(werr.isnan, np.isnan(gerr))
    assert (~w.isnan[..., 0]).mean() > min_valid
    wv, gv, we, ge = w.val, w.at(got), werr.val, werr.at(gerr)
    ok = np.isfinite(wv[:, 0])
    assert np.abs(wv[ok][:, :2] - gv[ok][:, :2]).max() < 1e-9
    assert np.abs(wv[ok][:, 2] - gv[ok][:, 2]).max() < 1e-6
    assert np.abs(we[ok] - ge[ok]).max() < 1e-4


def synthetic_inputs(with_direct):
    rng = np.random.default_rng(5)
    h, w = 60, 90
    rpc1, rpc2 = _rpc(1, with_direct), _rpc(2, with_direct)
    disp = (rng.normal(0, 6, (h, w))).astype(np.float32)
    mask = (rng.random((h, w)) > 0.2).astype(np.float32)
    H1, H2, bbx = _geometry()
    mo = (rng.random((int(bbx[3] - bbx[2]) + 1, int(bbx[1] - bbx[0]) + 1)) > 0.1).astype(np.float32)
    return disp, mask, mo, H1, H2, rpc1, rpc2, bbx


def real_inputs():
    """Real cameras: the RPCs of the reference's Pleiades fixture, its rectifying homographies and its shipped disparity map"""
    import make_golden_real_pair
    from s2p_b200.triangulation import rpc_from_geotiff_tag
    z = make_golden_real_pair.load()
    rpc1, rpc2 = rpc_from_geotiff_tag(z["rpc1"]), rpc_from_geotiff_tag(z["rpc2"])
    disp = z["rectified_disp"][100:260, 120:360].copy()
    # the rectified crop starts at (120, 100): move the origin into the homographies
    T = np.array([[1, 0, -120.0], [0, 1, -100.0], [0, 0, 1]])
    H1, H2 = T @ z["H1"], T @ z["H2"]
    mask = np.isfinite(disp).astype(np.float32)
    disp = np.nan_to_num(disp)
    bbx = (0.0, 1023.0, 0.0, 1023.0)
    mo = np.ones((1024, 1024), np.float32)
    mo[300:340, 500:560] = 0          # a hole in the image-domain mask
    return (disp, mask, mo, H1, H2, rpc1, rpc2, bbx), z


def triangulation_reference(oracle, key, args):
    def run():
        out, err = oracle.ref_disp_to_lonlatalt(*args)
        return {"lonlatalt": out, "err": err}
    return RR.reference_samples("disp_to_lonlatalt/" + key, run)


@pytest.mark.parametrize("with_direct", [False, True])
def test_matches_reference_library(engine, oracle, with_direct):
    from s2p_b200.triangulation import disp_to_lonlatalt
    args = synthetic_inputs(with_direct)
    want = triangulation_reference(oracle, "synthetic_direct=%d" % with_direct, args)
    got, gerr = disp_to_lonlatalt(*args, engine=engine)
    _assert_matches(got, gerr, want, 0.3)


def test_real_rpc_real_disparity(engine, oracle):
    """Real cameras: the RPCs of the reference's Pleiades fixture (tests/data/input_pair/img_0{1,2}.tif, RPCCoefficientTag,
    ground->image polynomials only, so every localisation runs the Newton iteration of c/rpc.c:378-411), its rectifying
    homographies and its shipped disparity map (tests/golden/real_pair*.npz), against the reference library."""
    from s2p_b200.triangulation import disp_to_lonlatalt
    args, z = real_inputs()
    want = triangulation_reference(oracle, "real", args)
    got, gerr = disp_to_lonlatalt(*args, engine=engine)
    _assert_matches(got, gerr, want, 0.5)
    # plausibility: the fixture is over the Reunion island area of the RPC offsets, altitudes within the RPC's height range
    assert abs(np.nanmedian(got[..., 0]) - z["rpc1"][5]) < 0.2 and abs(np.nanmedian(got[..., 1]) - z["rpc1"][4]) < 0.2
