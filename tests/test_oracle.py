"""CPU tests of the oracle (test infrastructure): the C restatement against the golden vectors
(outputs of the unmodified reference binary) and against the stored outputs of that binary and of the
reference's other programs on many more cases (tests/golden/reference_runs.py).  Bit-exact."""
import os
import subprocess
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
import make_golden as G  # noqa: E402
import reference_runs as RR  # noqa: E402
from util import nmismatch, same  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.mark.parametrize("name", sorted(G.CASES))
def test_port_matches_golden(oracle, name):
    ref, sec, dmin, dmax, kw = G.inputs(name)
    g = np.load(os.path.join(GOLD, name + ".npz"))
    algo, kw = G.split_kw(kw)
    wl, wr = G.weights_for(name) or (None, None)
    if algo == "mgm_multi":
        d, c, dr = oracle.port.mgm_multi(ref, sec, dmin, dmax, oracle.mgm_multi_params(dct_shift=1, **kw), wl, wr)
    else:
        d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params(dct_shift=1, **kw), wl, wr)
    assert same(d, g["disp"]), "%d px differ" % nmismatch(d, g["disp"])
    assert np.array_equal(c.astype(np.uint8), g["conf"])
    assert same(dr, g["dispR"])


@pytest.mark.parametrize("name", ["plain", "wide", "nan_ref", "tsgm4_o4", "census3", "real"])
def test_identity_shift_equals_dct_shift_without_nodata(oracle, name):
    """The reference pushes the matched image of each view through a DCT round trip even for a zero
    shift (mgm_costvolume.cc:23-60).  That is the identity except on exactly-zero pixels (NaN -> 0), whose
    value then depends on the FFT library's rounding noise.  Without no-data pixels the product's identity
    shift reproduces the reference bit for bit; with no-data in the reference image only, the right view
    (which matches against the shifted reference image) may differ near the no-data area, while the
    left disparity and the confidence of this fixture do not."""
    ref, sec, dmin, dmax, kw = G.inputs(name)
    g = np.load(os.path.join(GOLD, name + ".npz"))
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, oracle.mgm_params(dct_shift=0, **kw))
    assert same(d, g["disp"]) and np.array_equal(c.astype(np.uint8), g["conf"])
    if name != "nan_ref":
        assert same(dr, g["dispR"])


def test_roundtrip_flag_rule(oracle):
    """The engine only recomputes, through the DCT round trip, the pixels with |x| <= rowmax * n * 2^-24 (rows without such a
    pixel are left alone): s2p_b200/csrc/dct_kernels.cuh.  Check the claim behind that rule against the full round trip of the
    oracle: every other pixel returns to its float32 value.  Dynamic ranges from 12-bit imagery to 1e7:1, widths up to 2048."""
    import ctypes
    L = oracle.lib()
    rng = np.random.default_rng(1)
    changed = 0
    for n in (64, 200, 777, 1024, 2048):
        for kind in range(6):
            h = 12
            if kind == 0: x = rng.integers(0, 4096, (h, n)).astype(np.float32)
            elif kind == 1: x = rng.uniform(0, 65535, (h, n)).astype(np.float32)
            elif kind == 2: x = np.exp(rng.normal(0, 4, (h, n))).astype(np.float32)
            elif kind == 3: x = rng.uniform(0, 1, (h, n)).astype(np.float32)
            elif kind == 4: x = (rng.integers(0, 4096, (h, n)) * (rng.random((h, n)) < 0.5)).astype(np.float32)
            else:
                x = rng.uniform(-1000, 1000, (h, n)).astype(np.float32)
                x[:, :n // 10] = 0
                x[:, -n // 7:] = 0
            y = np.empty_like(x)
            L.orc_shift(oracle._p(x), oracle._p(y), n, h, ctypes.c_float(0.0), 1)
            thr = (np.abs(x).max(axis=1, keepdims=True) * np.float32(n * 2.0 ** -24)).astype(np.float32)
            unflagged = np.abs(x) > thr
            assert np.array_equal(y[unflagged], x[unflagged]), (n, kind)
            changed += int((y != x).sum())
    assert changed > 1000        # the round trip does move the flagged pixels


def _key(prefix, **kw):
    return prefix + "/" + ",".join("%s=%s" % (k, kw[k]) for k in sorted(kw))


def _outputs(r, *names):
    return {n: r[n] for n in names}


def _check(got, want):
    bad = RR.mismatches(got, want)
    assert not bad, "; ".join(bad)


@pytest.mark.parametrize("kw", [dict(), dict(tsgm=1), dict(tsgm=2), dict(tsgm=4), dict(ndir=4), dict(ndir=2),
                                dict(census_win=3), dict(census_win=7), dict(median=0, lr_mode=0, refine=0), dict(median=2),
                                dict(mindiff=1.0)])
def test_port_matches_reference_binary(oracle, kw):
    from s2p_b200.synth import make_pair
    h, w, dmin, dmax = 44, 72, -9, 10
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=33, nan_border=0.05)
    P = oracle.mgm_params(dct_shift=1, **kw)
    want = RR.reference_digests(_key("mgm", **kw), lambda: _outputs(oracle.run_ref(ref, sec, dmin, dmax, P, threads=1), "disp", "conf", "dispR"))
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, P)
    _check(dict(disp=d, conf=c, dispR=dr), want)


def test_port_cost_volume_matches_reference_dump(oracle):
    from s2p_b200.synth import make_pair
    h, w, dmin, dmax = 30, 64, -7, 9
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=7)
    P = oracle.mgm_params(dct_shift=1, median=0, lr_mode=0, refine=0)

    def run():
        r = oracle.run_ref(ref, sec, dmin, dmax, P, extra_env={"DUMP_COSTVOLUME": "1"})
        vol, dm = oracle.read_costvolume_dump(os.path.join(r["workdir"], "costvolume_left.dat"))
        assert dm == dmin
        return {"costvolume": vol}
    want = RR.reference_digests("costvolume_dump", run)
    lo = np.full((h, w), dmin, np.int32)
    hi = np.full((h, w), dmax, np.int32)
    C = oracle.port.costvolume(ref, sec, lo, hi, dmin, dmax - dmin + 1, dct_shift=1)
    _check({"costvolume": C}, want)


@pytest.mark.parametrize("kw", [dict(), dict(subpix=1), dict(scales=1), dict(lr_mode=2), dict(remove_small_cc=0, tsgm=3)])
def test_port_mgm_multi_matches_reference_binary(oracle, kw):
    from s2p_b200.synth import make_pair
    h, w, dmin, dmax = 112, 140, -14, 17
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=55, nan_border=0.04)
    P = oracle.mgm_multi_params(dct_shift=1, **kw)
    want = RR.reference_digests(_key("mgm_multi", **kw),
                                lambda: _outputs(oracle.run_ref(ref, sec, dmin, dmax, P, threads=1), "disp", "conf", "dispR"))
    d, c, dr = oracle.port.mgm_multi(ref, sec, dmin, dmax, P)
    _check(dict(disp=d, conf=c, dispR=dr), want)


def test_reference_sample_pair(oracle):
    """The reference's own shipped rectified pair (3rdparty/mgm_multi/matlab/data/rectified_{ref,sec}.tif, 279x271 with two NaN
    pixels): its top-left 160x120 crop, stored in tests/golden/sample_pair.npz."""
    z = np.load(os.path.join(GOLD, "sample_pair.npz"))
    a, b = z["ref"], z["sec"]
    P = oracle.mgm_params(dct_shift=1)
    want = RR.reference_digests("sample_pair", lambda: _outputs(oracle.run_ref(a, b, -22, 19, P), "disp", "conf", "dispR"))
    d, c, dr = oracle.port.mgm(a, b, -22, 19, P)
    _check(dict(disp=d, conf=c, dispR=dr), want)


def _lsd_like_weights(shape, seed, ones=0.6):
    rng = np.random.default_rng(seed)
    x = rng.uniform(0, 255, shape)
    w = np.maximum(((255 - x) / 255) ** 2, 0.1).astype(np.float32)
    w[rng.random(shape) < ones] = 1.0
    return w


@pytest.mark.parametrize("cost,kw", [(1, {}), (2, {"tsgm": 4}), (3, {"census_win": 3}), (3, {}), (3, {"census_win": 7}), (4, {}), (5, {"ndir": 4})])
def test_port_distances_match_reference_binary(oracle, cost, kw):
    """-t ad | sd | ncc | btad | btsd (mgm_costvolume.h:186-197), NaN-free and with no-data strips"""
    from s2p_b200.synth import make_pair
    h, w, dmin, dmax = 40, 66, -9, 8
    for nanb in (0.0, 0.06):
        ref, sec, _ = make_pair(h, w, dmin, dmax, seed=61 + cost, nan_border=nanb)
        P = oracle.mgm_params(dct_shift=1, cost=cost, **kw)
        want = RR.reference_digests(_key("distance", cost=cost, nan_border=nanb, **kw),
                                    lambda: _outputs(oracle.run_ref(ref, sec, dmin, dmax, P, threads=1), "disp", "conf", "dispR"))
        d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, P)
        _check(dict(disp=d, conf=c, dispR=dr), want)


@pytest.mark.parametrize("kw", [dict(tsgm=1), dict(tsgm=2), dict(tsgm=3), dict(tsgm=4), dict(tsgm=4, ndir=4), dict(tsgm=3, cost=1),
                                dict(tsgm=3, P1=7.0, P2=33.3)])
def test_port_weights_match_reference_binary(oracle, kw):
    """-wl / -wr with penalties whose products with the weights are inexact: pins how the reference build rounds
    x + P*w for each of the four neighbours (orc_fma_mask in oracle/mgm_oracle.c)"""
    from s2p_b200.synth import make_pair
    h, w, dmin, dmax = 48, 70, -10, 9
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=71)
    wl, wr = _lsd_like_weights((h, w), 1), _lsd_like_weights((h, w), 2, 0.3)
    kw = dict(dict(P1=12.0, P2=48.0), **kw)
    P = oracle.mgm_params(dct_shift=1, **kw)
    want = RR.reference_digests(_key("weights", **kw),
                                lambda: _outputs(oracle.run_ref(ref, sec, dmin, dmax, P, threads=1, wl=wl, wr=wr), "disp", "conf", "dispR"))
    d, c, dr = oracle.port.mgm(ref, sec, dmin, dmax, P, wl, wr)
    _check(dict(disp=d, conf=c, dispR=dr), want)


@pytest.mark.parametrize("kw,weighted", [(dict(P1=12.0, P2=48.0, median=1), True), (dict(cost=1), False), (dict(cost=3, subpix=1), False)])
def test_port_mgm_multi_options_match_reference_binary(oracle, kw, weighted):
    """what algo == 'mgm_multi_lsd' runs, and mgm_multi with another distance (half-pixel pass on the images)"""
    from s2p_b200.synth import make_pair
    h, w, dmin, dmax = 112, 140, -14, 17
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=81)
    wl, wr = (_lsd_like_weights((h, w), 3, 0.7), _lsd_like_weights((h, w), 4, 0.7)) if weighted else (None, None)
    P = oracle.mgm_multi_params(dct_shift=1, **kw)
    want = RR.reference_digests(_key("mgm_multi_options", weighted=weighted, **kw),
                                lambda: _outputs(oracle.run_ref(ref, sec, dmin, dmax, P, threads=1, wl=wl, wr=wr), "disp", "conf", "dispR"))
    d, c, dr = oracle.port.mgm_multi(ref, sec, dmin, dmax, P, wl, wr)
    _check(dict(disp=d, conf=c, dispR=dr), want)


def test_fuzz_sample_against_reference_binary(oracle):
    """A fixed sample of scripts/fuzz_oracle.py (random shapes, ranges, every parameter incl. MINDIFF, distances,
    weights, mgm and mgm_multi): the port must equal the binary on all of them."""
    import fuzz_oracle
    bad = []
    for case in fuzz_oracle.cases(24, 7):
        def run():
            try:
                r = oracle.run_ref(case["ref"], case["sec"], case["dmin"], case["dmax"], case["P"], threads=1, wl=case["wl"], wr=case["wr"])
            except subprocess.CalledProcessError:
                return None          # the reference refuses the case: nothing to compare, as in scripts/fuzz_oracle.py
            return _outputs(r, "disp", "conf", "dispR")
        want = RR.reference_digests("fuzz_7/%d" % case["it"], run)
        if want is None:
            continue
        fn = oracle.port.mgm_multi if case["multi"] else oracle.port.mgm
        d, c, dr = fn(case["ref"], case["sec"], case["dmin"], case["dmax"], case["P"], case["wl"], case["wr"])
        bad += ["case %d (%s): %s" % (case["it"], case["desc"], m) for m in RR.mismatches(dict(disp=d, conf=c, dispR=dr), want)]
    assert not bad, "\n".join(bad)


@pytest.mark.parametrize("shape,dmin,dmax,seed", [((60, 100), -11, 12, 0), ((90, 140), -20, 20, 1), ((41, 77), -5, 30, 2), ((33, 50), 0, 9, 3)])
def test_rejection_mask_port_matches_reference_programs(oracle, shape, dmin, dmax, seed):
    """create_rejection_mask (s2p/block_matching.py:18-32): the port against the reference's own plambda / backflow / plambda
    chain (c/plambda.c, c/backflow.c + bicubic.c + getpixel.c compiled in place as oracle/_ref/{plambda,backflow}), on tiles
    with no-data in both images, NaN disparities and disparities pointing outside the image."""
    from s2p_b200.synth import make_pair
    h, w = shape
    rng = np.random.default_rng(seed)
    ref, sec, gt = make_pair(h, w, dmin, dmax, seed=seed, nan_border=0.08)
    d = gt + rng.uniform(-0.7, 0.7, gt.shape).astype(np.float32)
    d[rng.random(d.shape) < 0.1] = np.nan
    d[:, :3] -= 7.3                   # backflow samples outside the image (getsample_0: zero outside)
    d[:, -3:] += 6.6
    want = RR.reference_digests("rejection_mask/%d" % seed, lambda: {"mask": oracle.ref_rejection_mask(d, ref, sec)})
    _check({"mask": oracle.port.rejection_mask(d, ref, sec)}, want)


@pytest.mark.parametrize("multi,shape,dmin,dmax,nanb,kw", [
    (False, (40, 70), -9, 10, 0.05, {}), (False, (30, 50), -3, 4, 0.1, dict(tsgm=4, census_win=3)), (False, (33, 60), -20, 5, 0.0, dict(refine=2)),
    (True, (110, 140), -12, 14, 0.0, {}), (True, (120, 150), -10, 9, 0.05, dict(subpix=1))])
def test_pkr_confidence_port_matches_reference_binary(oracle, multi, shape, dmin, dmax, nanb, kw):
    """-confidence_pkrL / -confidence_pkrR (compute_PKR_confidence, mgm_costvolume.cc:199-214) of mgm and mgm_multi; in
    mgm_multi the images written are the ZOOM = 1 call's (the SUBPIX pass has its own `param`, main_mgm_multi.cc:207)."""
    from s2p_b200.synth import make_pair
    h, w = shape
    ref, sec, _ = make_pair(h, w, dmin, dmax, seed=h, nan_border=nanb)
    P = oracle.mgm_multi_params(**kw) if multi else oracle.mgm_params(**kw)
    want = RR.reference_digests(_key("pkr", multi=multi, h=h, **kw),
                                lambda: _outputs(oracle.run_ref(ref, sec, dmin, dmax, P, want_pkr=True), "disp", "pkrL", "pkrR"))
    d, c, dr, pl, pr = oracle.port.mgm_pkr(ref, sec, dmin, dmax, P, multi=multi)
    _check(dict(disp=d, pkrL=pl, pkrR=pr), want)
