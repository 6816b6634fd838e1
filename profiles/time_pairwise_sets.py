"""Many independent image sets, pairwise: one aps_feature_matching_pairwise_sets call against one featureMatchingPairwise
call per set.

    python profiles/time_pairwise_sets.py [reps]

Batches: one C5 ring alone (30 x 4096 KAZE-64), synth config 5 split into its 10 rings of 30 images, two small-set
batches (64 sets of 6 x 300 rows, 300 sets of 3 x 200 rows, KAZE-64) and 16 binary sets of 6 x 2000 ORB-256 rows; each
with Matchingmethod 'Exhaustive' and with 'Approximate' / 'subsetpdist2' (subset 12000, so every image searches all
rows of its partner).  Threshold 1.5 (float) / 40 (binary), ratio 0.7, as bench.py's c5.  Both variants end with every
list on the host (the Python API's nested lists with metric); the time is the median of `reps` calls after one warm-up
call; the lists and metrics of both variants are compared in the same run.  Prints the card and its power limit."""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402


def small_sets(aps, B, shape, seed, kind="kaze", D=64):
    kp = max(300, max(shape))
    return [[im[:c] for im, c in zip(aps.synth.synth_descriptors(kind, len(shape), kp, D, seed + b), shape)]
            for b in range(B)]


def median_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def same_lists(x, y, n):
    (xm, xd), (ym, yd) = x, y
    for i in range(n):
        for j in range(n):
            a, b = np.asarray(xm[i][j]), np.asarray(ym[i][j])
            if a.shape != b.shape or not np.array_equal(a, b) or (xd[i][j] is None) != (yd[i][j] is None):
                return False
            if xd[i][j] is not None and not np.array_equal(xd[i][j], yd[i][j]):
                return False
    return True


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    aps = ge.load_package()
    ctx = aps._lib.default_context()
    c5, _ = aps.synth.make_config(5)
    cases = [("1 x (30 x 4096)", [c5[:30]], 1.5),
             ("C5 as 10 rings", [c5[30 * r:30 * r + 30] for r in range(10)], 1.5),
             ("64 x (6 x 300)", small_sets(aps, 64, [300] * 6, 300), 1.5),
             ("300 x (3 x 200)", small_sets(aps, 300, [200] * 3, 400), 1.5),
             ("16 x ORB 6 x 2000", [[aps.binaryFeatures(m) for m in s]
                                    for s in small_sets(aps, 16, [2000] * 6, 500, "orb", 32)], 40.0)]
    print(f"{'batch':>18} {'method':>13} {'pairs':>7} {'batched ms':>11} {'per-set ms':>11} {'speed-up':>8}  lists",
          flush=True)
    for method in ("Exhaustive", "subsetpdist2"):
        for name, sets, thr in cases:
            inp = {"Matchingmethod": "Exhaustive", "Matchingthreshold": thr, "Ratiothreshold": 0.7,
                   "useMATLABFeatureMatch": 0}
            if method != "Exhaustive":
                inp.update(Matchingmethod="Approximate", ApproxFloatNNMethod=method)
            nums = [len(s) for s in sets]
            res = {}
            tb = median_ms(lambda: res.__setitem__("b", aps.featureMatchingPairwiseSets(inp, sets, nums, ctx=ctx,
                                                                                       return_metric=True)), reps)
            ts = median_ms(lambda: res.__setitem__("s", [aps.featureMatchingPairwise(inp, s, n, ctx=ctx, return_metric=True)
                                                         for s, n in zip(sets, nums)]), reps)
            same = all(same_lists(x, y, n) for x, y, n in zip(res["b"], res["s"], nums))
            pairs = sum(n * (n - 1) // 2 for n in nums)
            print(f"{name:>18} {method:>13} {pairs:>7} {tb[0]:>11.2f} {ts[0]:>11.2f} {ts[0] / tb[0]:>8.2f}  "
                  f"{'identical' if same else 'DIFFER'}   (batched min/max {tb[1]:.2f}/{tb[2]:.2f}, "
                  f"per-set min/max {ts[1]:.2f}/{ts[2]:.2f})", flush=True)


if __name__ == "__main__":
    main()
