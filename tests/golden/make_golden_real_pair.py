"""Regenerates tests/golden/real_pair.npz from fixtures the reference ships for its own tests
(/root/reference/tests/data/input_pair/img_0{1,2}.tif, tests/data/input_triangulation/pair_1/{H_ref,H_sec}.txt,
rectified_ref.tif, rectified_disp.tif): real Pleiades imagery through the whole hot path.

* rectified_ref.tif IS homography(img_01.tif, H_ref.txt) at 503 x 425: a reference-held golden of the rectification warp.
* rectified_disp.tif is the reference's disparity for that pair (its rectified_sec.tif is not shipped: it is rebuilt by
  warping img_02.tif with H_sec.txt, and the matcher runs on [-41, 30]).

Only the source crops the two warps need are stored (uint16), with their offsets.  The arrays are split over three files
(real_pair.npz, real_pair_rectified_ref.npz, real_pair_rectified_disp.npz) that each stay under 1 MB; load() merges them.  The script checks the fixture with the
CPU oracles before writing: the reference resampler compiled in place reproduces rectified_ref.tif, and the reference
`mgm` on the rebuilt pair reproduces rectified_disp.tif to <= 0.25 px on > 99.5 % of the pixels.
    python tests/golden/make_golden_real_pair.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = "/root/reference/tests/data"
W, H = 503, 425
DMIN, DMAX = -41, 30


HERE = os.path.dirname(os.path.abspath(__file__))
RECTIFIED = ("rectified_ref", "rectified_disp")


def load():
    """-> {name: array} of the whole fixture"""
    z = dict(np.load(os.path.join(HERE, "real_pair.npz")))
    for name in RECTIFIED:
        z[name] = np.load(os.path.join(HERE, "real_pair_%s.npz" % name))[name]
    return z


def crop_for(Hm, img, w, h, margin=8):
    from s2p_b200.common import needed_roi
    x, y, rw, rh = needed_roi(Hm, w, h)
    x0, y0 = max(0, x - margin), max(0, y - margin)
    x1, y1 = min(img.shape[1], x + rw + margin), min(img.shape[0], y + rh + margin)
    return img[y0:y1, x0:x1], (x0, y0)


def compensate(Hm, xy):
    return np.asarray(Hm, np.float64) @ np.array([[1, 0, xy[0]], [0, 1, xy[1]], [0, 0, 1.0]])


def main():
    from oracle import oracle as O
    from s2p_b200 import rasterio_compat as rio
    im1 = rio.read_band(os.path.join(REF, "input_pair", "img_01.tif"))
    im2 = rio.read_band(os.path.join(REF, "input_pair", "img_02.tif"))
    H1 = np.loadtxt(os.path.join(REF, "input_triangulation", "pair_1", "H_ref.txt"))
    H2 = np.loadtxt(os.path.join(REF, "input_triangulation", "pair_1", "H_sec.txt"))
    rect_ref = rio.read_band(os.path.join(REF, "input_triangulation", "pair_1", "rectified_ref.tif"))
    rect_disp = rio.read_band(os.path.join(REF, "input_triangulation", "pair_1", "rectified_disp.tif"))
    assert rect_ref.shape == (H, W) and rect_disp.shape == (H, W)
    c1, xy1 = crop_for(H1, im1, W, H)
    c2, xy2 = crop_for(H2, im2, W, H)
    assert np.array_equal(c1, np.round(c1)) and c1.max() < 65536
    # self-check with the CPU oracles
    w1 = O.run_ref_homography(c1, compensate(H1, xy1), W, H)
    nanmis = int((np.isnan(w1) != np.isnan(rect_ref)).sum())
    both = np.isfinite(w1) & np.isfinite(rect_ref)
    err = float(np.abs(w1[both] - rect_ref[both]).max())
    print("warp vs rectified_ref.tif: NaN mismatches %d, max |d| %.4f of range %.1f" % (nanmis, err, np.nanmax(rect_ref)))
    w2 = O.run_ref_homography(c2, compensate(H2, xy2), W, H)
    r = O.run_ref(rect_ref, w2, DMIN, DMAX, O.mgm_params(), threads=1)
    both = np.isfinite(r["disp"]) & np.isfinite(rect_disp)
    d = np.abs(r["disp"][both] - rect_disp[both])
    print("reference mgm vs rectified_disp.tif: %.2f %% within 0.25 px, median %.2g, NaN mask differs on %.2f %%" % (
        100 * (d <= 0.25).mean(), np.median(d), 100 * (np.isnan(r["disp"]) != np.isnan(rect_disp)).mean()))
    # the cameras: the RPCCoefficientTag (50844) of the two GeoTIFFs, 92 doubles each
    from PIL import Image
    rpcs = []
    for name in ("img_01.tif", "img_02.tif"):
        with Image.open(os.path.join(REF, "input_pair", name)) as im:
            rpcs.append(np.array(im.tag_v2[50844], np.float64))
    assert rpcs[0].size == 92 and rpcs[1].size == 92
    np.savez_compressed(os.path.join(HERE, "real_pair.npz"), crop1=c1.astype(np.uint16), xy1=np.array(xy1), crop2=c2.astype(np.uint16),
                        xy2=np.array(xy2), H1=H1, H2=H2, rpc1=rpcs[0], rpc2=rpcs[1])
    for name, a in zip(RECTIFIED, (rect_ref, rect_disp)):
        np.savez_compressed(os.path.join(HERE, "real_pair_%s.npz" % name), **{name: a})


if __name__ == "__main__":
    main()
