"""TEST INFRASTRUCTURE ONLY -- numpy restatement of s2p.fusion.merge_n's arithmetic (s2p/fusion.py:16-68).

`merge_ref` runs the REFERENCE's own `average_if_close`, extracted from its s2p/fusion.py (S2PB_FUSION_REFERENCE, default:
the reference tree beside the repository) when that file is present (the module itself cannot be imported here: it needs rasterio), through np.apply_along_axis
exactly as merge_n does; `merge_port` is the vectorised restatement used where the reference is absent.
"""
import ast
import os
import warnings

import numpy as np

REF = os.environ.get("S2PB_FUSION_REFERENCE") or os.path.join(os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))),
                                                              "reference", "s2p", "fusion.py")


def reference_average_if_close():
    """-> the reference's function object, or None when the reference's fusion.py is absent."""
    if not os.path.exists(REF):
        return None
    tree = ast.parse(open(REF).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "average_if_close"][0]
    ns = {"np": np}
    exec(compile(ast.Module([fn], []), REF, "exec"), ns)
    return ns["average_if_close"]


def _stack(rasters, offsets, sub_f32):
    """x[:, :, i] = f.read(1) - offsets[i] (s2p/fusion.py:45-49) with offsets[i] the 0-d float64 array np.loadtxt returns
    (s2p/__init__.py:371-374).  sub_f32=None: let the installed NumPy evaluate that very expression; True / False: force the
    NumPy < 2 (float32, value-based casting) / NumPy >= 2 (float64, NEP 50) behaviour."""
    h, w = np.asarray(rasters[0]).shape
    x = np.empty((h, w, len(rasters)))
    for i, (r, o) in enumerate(zip(rasters, offsets)):
        r = np.asarray(r, np.float32)
        if sub_f32 is None:
            x[:, :, i] = r - np.array(float(o))
        elif sub_f32:
            x[:, :, i] = r - np.float32(o)
        else:
            x[:, :, i] = r.astype(np.float64) - float(o)
    return x


def merge_ref(rasters, offsets, threshold, sub_f32=None):
    f = reference_average_if_close()
    x = _stack(rasters, offsets, sub_f32)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        avg = np.apply_along_axis(f, 2, x, threshold)
    avg += np.mean(offsets)
    return avg.astype("float32")


def merge_port(rasters, offsets, averaging="average_if_close", threshold=1, sub_f32=None):
    x = _stack(rasters, offsets, sub_f32)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if averaging == "average_if_close":
            spread = np.nanmax(x, axis=2) - np.nanmin(x, axis=2)
            avg = np.where(spread > threshold, np.nan, np.nanmedian(x, axis=2))
        else:       # the reference goes through apply_along_axis: one 1-D call per pixel (s2p/fusion.py:53-55)
            avg = np.apply_along_axis(getattr(np, averaging.split(".")[1]), 2, x)
    avg = avg + np.mean(offsets)
    return avg.astype("float32")
