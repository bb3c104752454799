"""Fuzz the CPU oracle (oracle/liboracle.so) against the unmodified reference binaries (oracle/_ref) on random
shapes, ranges and parameters.  CPU only; needs oracle/_ref (make -C oracle ref).  usage: python scripts/fuzz_oracle.py [N] [seed]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np

from oracle import oracle as O
from s2p_b200.synth import make_pair


def differ(a, b):
    return int((~((a == b) | (np.isnan(a) & np.isnan(b)))).sum())


def cases(n, seed):
    """-> the n random cases of `seed`, as dicts (it, multi, ref, sec, dmin, dmax, P, wl, wr, desc)"""
    rng = np.random.default_rng(seed)
    for it in range(n):
        multi = rng.random() < 0.3
        h, w = (int(rng.integers(101, 140)), int(rng.integers(101, 170))) if multi else (int(rng.integers(6, 60)), int(rng.integers(8, 90)))
        dmin = int(rng.integers(-30, 10))
        dmax = dmin + int(rng.integers(2, 40))
        kw = dict(ndir=int(rng.choice([2, 4, 8])), tsgm=int(rng.integers(1, 5)), census_win=int(rng.choice([3, 5, 7])),
                  P1=float(rng.choice([8.0, 12.0, 5.5])), P2=float(rng.choice([32.0, 48.0, 41.0])), median=int(rng.integers(0, 3)),
                  lr_mode=int(rng.integers(0, 2)), refine=int(rng.choice([0, 1, 1, 2])), cost=int(rng.choice([0, 0, 0, 1, 2, 3, 4, 5])),
                  mindiff=float(rng.choice([-1.0, -1.0, 1.0])), dct_shift=1)
        if kw["refine"] == 2:
            kw["refine"] = 1        # the parabola fit is only pinned to 1 ulp (DESIGN.md section 4)
        nanb = float(rng.choice([0.0, 0.0, 0.05]))
        if multi:
            kw.update(subpix=int(rng.choice([1, 2])), scales=int(rng.choice([1, 3, 6])), remove_small_cc=int(rng.choice([0, 25])),
                      lr_mode=int(rng.integers(0, 3)))
            P = O.mgm_multi_params(**kw)
        else:
            P = O.mgm_params(**kw)
        ref, sec, _ = make_pair(h, w, dmin, dmax, seed=int(rng.integers(1 << 30)), nan_border=nanb)
        wl = wr = None
        if rng.random() < 0.4:
            def wt():
                x = rng.uniform(0, 255, (h, w))
                a = np.maximum(((255 - x) / 255) ** 2, 0.1).astype(np.float32)
                a[rng.random((h, w)) < 0.6] = 1.0
                return a
            wl, wr = wt(), wt()
        desc = "%s %s %d %d %s%s nan %s" % ("multi" if multi else "mgm", (h, w), dmin, dmax, kw, " weights" if wl is not None else "", nanb)
        yield dict(it=it, multi=multi, ref=ref, sec=sec, dmin=dmin, dmax=dmax, P=P, wl=wl, wr=wr, desc=desc)


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    bad = 0
    for c in cases(n, int(sys.argv[2]) if len(sys.argv) > 2 else 0):
        try:
            r = O.run_ref(c["ref"], c["sec"], c["dmin"], c["dmax"], c["P"], threads=1, wl=c["wl"], wr=c["wr"])
        except Exception as e:
            print(c["it"], "reference failed:", type(e).__name__, c["desc"])
            continue
        fn = O.port.mgm_multi if c["multi"] else O.port.mgm
        d, cf, dr = fn(c["ref"], c["sec"], c["dmin"], c["dmax"], c["P"], c["wl"], c["wr"])
        nd, nc, nr = differ(d, r["disp"]), differ(cf, r["conf"]), differ(dr, r["dispR"])
        if nd or nc or nr:
            bad += 1
            print(c["it"], "MISMATCH", (nd, nc, nr), c["desc"], flush=True)
    print("done: %d cases, %d with a mismatch" % (n, bad))


if __name__ == "__main__":
    main()
