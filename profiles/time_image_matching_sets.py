"""Many independent image sets, image matching: one imageMatchingSets call against one imageMatching call per set.

    python profiles/time_image_matching_sets.py [reps]

Batches (synth.synth_matched_keypoints rings, maxIter 500, maxDistance 5.5, confidence 99.9, m = 6): one C1-shaped set
(6 images x 2048 keypoints, image 4 empty), config 5 as its 10 rings of 30 images x 4096 keypoints, 64 sets of
6 x 300 keypoints and 300 sets of 3 x 200 keypoints.  Both variants end with every set's cells on the host (the Python
API's nested lists); the time is the median of `reps` calls after one warm-up call; the raw outputs of both variants
(pairs, offsets, model and inverse bits, inliers, n_inliers, accepted, draws_used) are compared in the same run.
Prints the card and its power limit."""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402

PARAMS = {"maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}
KEYS = ("pairs_lin", "pt_ptr", "n_inliers", "accepted", "draws_used", "inliers", "models", "models_inv")


def ring_sets(aps, B, n, kp, seed, empty=()):
    ns, kps, ms = [], [], []
    for b in range(B):
        k, m, _ = aps.synth.synth_matched_keypoints(n, kp, seed=seed + b)
        for e in empty:
            k[e] = np.zeros((0, 2))
            for j in range(n):
                m[e][j] = m[j][e] = np.zeros((0, 0))
        ns.append(n), kps.append(k), ms.append(m)
    return ns, kps, ms


def median_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def same(x, y):
    for k in KEYS:
        a, b = np.asarray(x[k]), np.asarray(y[k])
        if a.dtype == np.float64:
            a, b = a.view(np.uint64), b.view(np.uint64)
        if a.shape != b.shape or not np.array_equal(a, b):
            return False
    return True


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    aps = ge.load_package()
    ctx = aps._lib.default_context()
    cases = [("1 x C1", ring_sets(aps, 1, 6, 2048, 100, empty=(3,))),
             ("C5 as 10 rings", ring_sets(aps, 10, 30, 4096, 200)),
             ("64 x (6 x 300)", ring_sets(aps, 64, 6, 300, 300)),
             ("300 x (3 x 200)", ring_sets(aps, 300, 3, 200, 400))]
    print(f"{'batch':>16} {'pairs':>6} {'sets call ms':>13} {'per-set ms':>11} {'speed-up':>8}  outputs", flush=True)
    for name, (ns, kps, ms) in cases:
        res = {}

        def batched():
            aps.imageMatchingSets(PARAMS, ns, kps, ms, seed=1, ctx=ctx)
            res["b"] = list(aps.imageMatchingSets.last)

        def per_set():
            out = []
            for n, k, m in zip(ns, kps, ms):
                aps.imageMatching(PARAMS, n, k, m, seed=1, ctx=ctx)
                out.append(dict(aps.imageMatching.last))
            res["s"] = out

        tb = median_ms(batched, reps)
        ts = median_ms(per_set, reps)
        ok = all(same(x, y) for x, y in zip(res["b"], res["s"]))
        pairs = sum(len(d["pairs_lin"]) for d in res["b"])
        print(f"{name:>16} {pairs:>6} {tb[0]:>13.2f} {ts[0]:>11.2f} {ts[0] / tb[0]:>8.2f}  "
              f"{'identical' if ok else 'DIFFER'}   (sets call min/max {tb[1]:.2f}/{tb[2]:.2f}, "
              f"per-set min/max {ts[1]:.2f}/{ts[2]:.2f})", flush=True)


if __name__ == "__main__":
    main()
