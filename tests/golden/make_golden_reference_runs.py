"""Records tests/golden/reference_runs.json and reference_samples.npz (see reference_runs.py): the outputs of the unmodified
reference programs (oracle/_ref, built by `make -C oracle ref` from the reference sources) on every case of the tests that
compare with them, and sample_pair.npz, the crop of the reference's sample pair those tests read.  Needs the reference tree
(REF_ROOT, default ../reference beside the repository), no GPU.
    python tests/golden/make_golden_reference_runs.py [REF_ROOT]
"""
import os
import subprocess
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TESTS = os.path.dirname(HERE)
for p in (ROOT, TESTS, HERE):
    sys.path.insert(0, p)


def main():
    ref_root = os.path.abspath(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "..", "reference"))
    from oracle import oracle as O
    assert O.have_ref() and O.have_ref_mask() and O.have_ref_homography() and O.have_ref_morsi() and O.have_ref_triangulation(), \
        "build oracle/_ref first: make -C oracle ref"
    from s2p_b200 import rasterio_compat as rio
    src = os.path.join(ref_root, "3rdparty", "mgm_multi", "matlab", "data")
    np.savez_compressed(os.path.join(HERE, "sample_pair.npz"), ref=rio.read_band(os.path.join(src, "rectified_ref.tif"))[:120, :160],
                        sec=rio.read_band(os.path.join(src, "rectified_sec.tif"))[:120, :160])
    for f in ("reference_runs.json", "reference_samples.npz"):
        if os.path.exists(os.path.join(HERE, f)):
            os.remove(os.path.join(HERE, f))
    os.environ["S2PB_RECORD_REFERENCE"] = "1"
    # the CPU tests record their cases as they run; average_if_close is read from the reference tree
    env = dict(os.environ, S2PB_FUSION_REFERENCE=os.path.join(ref_root, "s2p", "fusion.py"))
    subprocess.run([sys.executable, "-m", "pytest", "-q", "-p", "no:cacheprovider", os.path.join(TESTS, "test_oracle.py"),
                    os.path.join(TESTS, "test_fusion.py") + "::test_port_matches_reference_function"], check=True, cwd=ROOT, env=env)
    # the GPU tests' cases: their reference halves, without a GPU
    import test_fusion
    import test_gpu_homography
    import test_gpu_parity
    import test_triangulation
    for case in test_gpu_parity.NODATA_CASES:
        test_gpu_parity.nodata_reference(O, *case)
    test_gpu_parity.rejection_mask_reference(O)
    for name in test_gpu_homography.CASES:
        test_gpu_homography.warp_reference(O, name)
    test_gpu_homography.dropin_reference(O)
    for with_direct in (False, True):
        test_triangulation.triangulation_reference(O, "synthetic_direct=%d" % with_direct,
                                                   test_triangulation.synthetic_inputs(with_direct))
    test_triangulation.triangulation_reference(O, "real", test_triangulation.real_inputs()[0])
    for radius in test_fusion.EROSION_RADII:
        test_fusion.erosion_reference(O, radius)


if __name__ == "__main__":
    main()
