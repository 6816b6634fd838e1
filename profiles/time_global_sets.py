"""Many independent image sets: one aps_feature_matching_global_sets call against one featureMatchingGlobal call per set.

    python profiles/time_global_sets.py [reps]

Sets are synth config 1 (6 images x 2048 SIFT-128, one image empty; "C1-sized") made distinct per set by a row
permutation and a +-1 integer perturbation (config 1 is integer-valued), 4 C2-sized sets (config 2, perturbed alike),
two small-set batches below the tensor path's size (64 sets of 6 x 300 rows, 300 sets of 3 x 200 rows) and 16 binary
sets of 6 x 20000 ORB-256 rows.  Both
variants end with every list on the host (the Python API's nested lists); the time is the median of `reps` calls after
one warm-up call; the lists of both variants are compared in the same run.  Prints the card and its power limit."""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402


def perturbed(desc, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    out = []
    for d in desc:
        if d.shape[0] == 0:
            out.append(d)
            continue
        d = d[rng.permutation(d.shape[0])]
        out.append(np.clip(d + rng.integers(-1, 2, d.shape), 0, 255).astype(np.float32))
    return out


def small_sets(aps, B, shape, seed):
    kp = max(300, max(shape))
    return [[im[:c] for im, c in zip(aps.synth.synth_descriptors("sift", len(shape), kp, 128, seed + b), shape)]
            for b in range(B)]


def median_ms(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), float(np.max(ts))


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    aps = ge.load_package()
    ctx = aps._lib.default_context()
    c1, p1 = aps.synth.make_config(1)
    c2, p2 = aps.synth.make_config(2)
    cases = [(f"{B} x C1", [perturbed(c1, 100 + b) for b in range(B)], p1) for B in (1, 16, 64, 256)]
    cases.append(("4 x C2", [perturbed(c2, 200 + b) for b in range(4)], p2))
    cases.append(("64 x (6 x 300)", small_sets(aps, 64, [300] * 6, 300), p1))
    cases.append(("300 x (3 x 200)", small_sets(aps, 300, [200] * 3, 400), p1))
    orb = [[aps.binaryFeatures(m) for m in aps.synth.synth_descriptors("orb", 6, 20000, 32, 500 + b)] for b in range(16)]
    cases.append(("16 x ORB 6 x 20000", orb, aps.synth.CONFIGS[4]))
    print(f"{'batch':>16} {'rows':>9} {'batched ms':>11} {'per-set ms':>11} {'speed-up':>8}  lists", flush=True)
    for name, sets, p in cases:
        inp = {"k": p["k"], "Ratiothreshold": p["ratio"]}
        nums = [len(s) for s in sets]
        res = {}
        tb = median_ms(lambda: res.__setitem__("b", aps.featureMatchingGlobalSets(inp, sets, nums, ctx=ctx)), reps)
        ts = median_ms(lambda: res.__setitem__("s", [aps.featureMatchingGlobal(inp, s, n, ctx=ctx)
                                                     for s, n in zip(sets, nums)]), reps)
        same = all(np.array_equal(np.asarray(x[i][j]), np.asarray(y[i][j])) and
                   np.asarray(x[i][j]).shape == np.asarray(y[i][j]).shape
                   for x, y, n in zip(res["b"], res["s"], nums) for i in range(n) for j in range(n))
        rows = sum(getattr(d, "Features", d).shape[0] for s in sets for d in s)
        print(f"{name:>16} {rows:>9} {tb[0]:>11.2f} {ts[0]:>11.2f} {ts[0] / tb[0]:>8.2f}  "
              f"{'identical' if same else 'DIFFER'}   (batched min/max {tb[1]:.2f}/{tb[2]:.2f}, "
              f"per-set min/max {ts[1]:.2f}/{ts[2]:.2f})", flush=True)


if __name__ == "__main__":
    main()
