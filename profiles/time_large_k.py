"""Global matching at k > 4: C2 (20 images x 8192 SIFT-128) through GlobalPlan at k = 4, 6, 8, 12, 13 with the auto
engine (tensor path for k <= 12, exact CUDA-core engine above), and at k = 8, 12 also with the exact engine.

The variants are alternated in one session (order reversed every run), `--runs` timed steps each after one warm-up
step.  A step is prepare + knn + filter + compact, timed with a device synchronise.  Per variant it prints the median
and range of the step time and of the k_knn_tc time (CUDA events, aps_ctx_tc_time), the rows the first completeness
proof left open and the rows the exact fallback searched, and checks that the kNN tables and match lists of the two
engines are byte-equal at k = 8 and 12.  The card's name, power limit and max SM clock are read in the same call.

    python profiles/time_large_k.py [--runs 5] [--config 2]
"""
from __future__ import annotations

import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--config", type=int, default=2)
    a = ap.parse_args()
    pkg = ge.load_package()
    print("card (name, power limit, max SM clock):", card(), flush=True)
    desc, c = pkg.synth.make_config(a.config)
    ctx = pkg.Context(0)
    ctx.enable_timing(True)
    variants = [(4, 0), (6, 0), (8, 0), (12, 0), (13, 0), (8, 1), (12, 1)]  # (k, engine: 0 auto, 1 exact)
    plans = {}
    for k, eng in variants:
        ctx.set_float_engine(eng)  # the engine is chosen when the plan is created
        plans[(k, eng)] = pkg.GlobalPlan(ctx, [d.shape[0] for d in desc], desc[0].shape[1], False, k)
        plans[(k, eng)].upload(desc)
    ctx.set_float_engine(0)
    F = plans[variants[0]].F
    print(f"config {a.config}: {c['n']} x {c['kp']} D={desc[0].shape[1]} F={F} ratio={c['ratio']}", flush=True)

    def step(v):
        plan = plans[v]
        ctx.synchronize()
        t0 = time.perf_counter()
        plan.prepare()
        plan.knn()
        plan.filter(c["ratio"])
        plan.compact()
        ctx.synchronize()
        ms = 1e3 * (time.perf_counter() - t0)
        tc_ms, launches = ctx.tc_time()
        st = ctx.last_stats()
        return dict(ms=ms, tc_ms=tc_ms, launches=launches, engine=st["engine"], fallback=st["fallback_rows"],
                    unproven=ctx.first_pass_unproven() if st["engine"] == "tcgen05" else 0)

    res = {v: [] for v in variants}
    for v in variants:
        step(v)  # warm-up: module load, allocations
    for r in range(a.runs):
        for v in (variants if r % 2 == 0 else variants[::-1]):
            res[v].append(step(v))
    for v in variants:
        rs = res[v]
        ms, tc = [x["ms"] for x in rs], [x["tc_ms"] for x in rs]
        tflops = 2.0 * desc[0].shape[1] * F * F / (statistics.median(tc) * 1e-3) / 1e12 if rs[0]["launches"] else 0.0
        print(f"k={v[0]:2d} engine={'auto ' if v[1] == 0 else 'exact'} ({rs[0]['engine']:7s}): step median "
              f"{statistics.median(ms):9.3f} ms range {min(ms):9.3f}-{max(ms):9.3f} | k_knn_tc median "
              f"{statistics.median(tc):7.3f} ms range {min(tc):7.3f}-{max(tc):7.3f} ({rs[0]['launches']} launches/step"
              f"{f', {tflops:.0f} TFLOP/s' if tflops else ''}) | first_pass_unproven {rs[-1]['unproven']} "
              f"fallback_rows {rs[-1]['fallback']} | n={len(rs)}", flush=True)
    for k in (8, 12):
        ta, tb = plans[(k, 0)].download_knn(), plans[(k, 1)].download_knn()
        ma, mb = plans[(k, 0)].download()[2:], plans[(k, 1)].download()[2:]
        same_knn = all(np.asarray(x).tobytes() == np.asarray(y).tobytes() for x, y in zip(ta, tb))
        same_m = all(np.asarray(x).tobytes() == np.asarray(y).tobytes() for x, y in zip(ma, mb))
        speed = statistics.median([x["ms"] for x in res[(k, 1)]]) / statistics.median([x["ms"] for x in res[(k, 0)]])
        print(f"k={k}: tensor vs exact engine: kNN tables {'byte-equal' if same_knn else 'DIFFER'}, match lists "
              f"{'byte-equal' if same_m else 'DIFFER'} ({len(ma[1])} rows); exact / tensor step time {speed:.1f}x",
              flush=True)
    for p in plans.values():
        p.close()


if __name__ == "__main__":
    main()
