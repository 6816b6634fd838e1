"""featureMatchingPairwise + imageMatching: one pairwiseImageMatchingSets call against the two-call chain
featureMatchingPairwiseSets -> imageMatchingSets, alternated in one run.

    python profiles/time_pairwise_image_matching.py [reps]

Batches (make_set of tests/test_gpu_global_image_matching.py: SIFT-like 128-dimensional descriptors on rings, 30% of
each image's rows shared with the previous image, keypoints of the shared rows related by a homography for 3 in 4
pairs; Matchingthreshold 1.5, Ratiothreshold 0.8, m = 6, maxIter 500, maxDistance 5.5, confidence 99.9): one
C1-shaped set (6 x 2048, image 4 empty), config 5's shape as 10 rings of 30 images x 4096 rows, config 5's shape as
one set (300 x 4096; SIFT-like rather than KAZE-64), 64 sets of 6 x 300 and 300 sets of 3 x 200, each with
Matchingmethod 'Exhaustive' and with 'Approximate' / 'subsetpdist2' (apsSubset 12000, so every image is matched
whole).  Both variants end with every set's allMatches, numMatches and
tforms on the host as the Python API returns them.  Each repetition runs the chain and the fused call back to back
(the order alternating); the times are the median (min / max) of `reps` repetitions after one warm-up of each.  The
outputs of both variants (allMatches, numMatches, tforms bits, pairs, offsets, n_inliers, accepted, draws_used, model
bits) are compared in the same run.  Prints the card, its power limit and its maximum SM clock."""
import os
import subprocess
import sys
import time

import numpy as np

HERE = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "tests"))
import __graft_entry__ as ge  # noqa: E402
from test_gpu_global_image_matching import make_set  # noqa: E402
from test_gpu_pairwise_image_matching import METHODS, PARAMS  # noqa: E402

KEYS = ("pairs_lin", "pt_ptr", "n_inliers", "accepted", "draws_used", "models", "models_inv")


def batch(aps, B, n, kp, seed, empty=()):
    rng = np.random.default_rng(seed)
    cells, kps = zip(*[make_set(aps, rng, n, kp, empty=empty) for _ in range(B)])
    return list(cells), list(kps), [n] * B


def bits(a):
    a = np.asarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def same(x, y, lx, ly):
    for (aA, aN, aT), (bA, bN, bT) in zip(x, y):
        n = aN.shape[0]
        if not np.array_equal(aN, bN):
            return False
        for i in range(n):
            for j in range(n):
                if not np.array_equal(np.asarray(aA[i][j]), np.asarray(bA[i][j])):
                    return False
                if (aT[i][j] is None) != (bT[i][j] is None) or (
                        aT[i][j] is not None and not np.array_equal(bits(aT[i][j]), bits(bT[i][j]))):
                    return False
    for a, b in zip(lx, ly):
        for k in KEYS:
            if k in b and not np.array_equal(bits(a[k]), bits(b[k])):
                return False
    return True


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    aps = ge.load_package()
    ctx = aps._lib.default_context()
    cases = [("1 x C1", lambda: batch(aps, 1, 6, 2048, 100, empty=(3,))),
             ("C5 as 10 rings", lambda: batch(aps, 10, 30, 4096, 200)),
             ("C5 (300 x 4096)", lambda: batch(aps, 1, 300, 4096, 250)),
             ("64 x (6 x 300)", lambda: batch(aps, 64, 6, 300, 300)),
             ("300 x (3 x 200)", lambda: batch(aps, 300, 3, 200, 400))]
    print(f"{'batch':>16} {'method':>12} {'pairs':>6} {'accepted':>8} {'fused ms':>9} {'chain ms':>9} {'speed-up':>8}"
          "  outputs", flush=True)
    for name, make in cases:
        cells, kps, ns = make()
        for method in ("Exhaustive", "subsetpdist2"):
            inp = dict(PARAMS, **METHODS[method])
            res = {}

            def fused():
                res["f"] = aps.pairwiseImageMatchingSets(inp, cells, ns, kps, seed=1, ctx=ctx)
                res["fl"] = list(aps.pairwiseImageMatchingSets.last)

            def chain():
                m = aps.featureMatchingPairwiseSets(inp, cells, ns, ctx=ctx)
                res["c"] = aps.imageMatchingSets(inp, ns, kps, m, seed=1, ctx=ctx)
                res["cl"] = list(aps.imageMatchingSets.last)

            fused(), chain()
            tf, tc = [], []
            for r in range(reps):
                for fn, ts in (((fused, tf), (chain, tc)) if r % 2 == 0 else ((chain, tc), (fused, tf))):
                    ctx.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    ts.append((time.perf_counter() - t0) * 1e3)
            ok = same(res["f"], res["c"], res["fl"], res["cl"])
            pairs = sum(len(d["pairs_lin"]) for d in res["fl"])
            acc = sum(int(d["accepted"].sum()) for d in res["fl"])
            mf, mc = float(np.median(tf)), float(np.median(tc))
            print(f"{name:>16} {method:>12} {pairs:>6} {acc:>8} {mf:>9.2f} {mc:>9.2f} {mc / mf:>8.2f}  "
                  f"{'identical' if ok else 'DIFFER'}   (fused min/max {min(tf):.2f}/{max(tf):.2f}, "
                  f"chain min/max {min(tc):.2f}/{max(tc):.2f})", flush=True)
        del cells, kps


if __name__ == "__main__":
    main()
