"""Old-versus-new benchmark in one GPU session: runs `bench.py --no-cpu-baseline --no-extra` of two built trees
alternately (old, new, old, new, ...; the order flips every round) and prints, per build and config, the median and
range of ms_per_step and roofline.kernel_ms, with the card's name, power limit and the clocks bench.py read.

    python profiles/ab_bench.py --old OLD_TREE --new NEW_TREE --runs 5 --configs c2 --out OUTDIR
    python profiles/ab_bench.py ... --dump c2,c6,c5   # first: one --dump-outputs run per build and config, compared

Each tree must already be built (__graft_entry__.build()).  Raw JSON lines go to OUTDIR/ab_<config>.jsonl.
"""
from __future__ import annotations

import argparse
import filecmp
import json
import os
import statistics
import subprocess
import sys


def run_bench(tree, config, extra=()):
    cmd = [sys.executable, os.path.join(tree, "bench.py"), "--config", config, "--no-cpu-baseline", "--no-extra", *extra]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    if r.returncode or not lines:
        raise SystemExit(f"{' '.join(cmd)} failed ({r.returncode}):\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}")
    return json.loads(lines[-1])


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def compare_dumps(a, b):
    names = sorted(set(os.listdir(a)) | set(os.listdir(b)))
    bad = [n for n in names if not (os.path.exists(os.path.join(a, n)) and os.path.exists(os.path.join(b, n))
                                    and filecmp.cmp(os.path.join(a, n), os.path.join(b, n), shallow=False))]
    return names, bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--old", required=True)
    ap.add_argument("--new", required=True)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--configs", default="c2")
    ap.add_argument("--dump", default="", help="configs whose --dump-outputs files are compared byte for byte")
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    trees = {"old": os.path.abspath(a.old), "new": os.path.abspath(a.new)}
    print("card (name, power limit, max SM clock):", card(), flush=True)
    for c in filter(None, a.dump.split(",")):
        dirs = {}
        for b, t in trees.items():
            dirs[b] = os.path.join(os.path.abspath(a.out), f"dump_{c}_{b}")
            line = run_bench(t, c, ("--dump-outputs", dirs[b]))
            print(f"dump {c} {b}: parity_check={line.get('parity_check')}", flush=True)
        names, bad = compare_dumps(dirs["old"], dirs["new"])
        print(f"dump {c}: {len(names)} files {names}, " + ("byte-identical" if not bad else f"DIFFER: {bad}"), flush=True)
    for c in filter(None, a.configs.split(",")):
        res = {"old": [], "new": []}
        with open(os.path.join(a.out, f"ab_{c}.jsonl"), "w") as f:
            for i in range(a.runs):
                for b in (("old", "new") if i % 2 == 0 else ("new", "old")):
                    line = run_bench(trees[b], c)
                    res[b].append(line)
                    f.write(json.dumps({"build": b, "run": i, **line}) + "\n")
                    f.flush()
                    print(f"{c} run {i} {b}: ms_per_step {line['ms_per_step']:.4f} kernel_ms "
                          f"{line.get('roofline', {}).get('kernel_ms', float('nan')):.4f} clocks {line.get('clocks')}", flush=True)
        for b in ("old", "new"):
            ms = [l["ms_per_step"] for l in res[b]]
            km = [l.get("roofline", {}).get("kernel_ms", float("nan")) for l in res[b]]
            print(f"{c} {b}: ms_per_step median {statistics.median(ms):.4f} range {min(ms):.4f}-{max(ms):.4f} | "
                  f"kernel_ms median {statistics.median(km):.4f} range {min(km):.4f}-{max(km):.4f} | n={len(ms)}",
                  flush=True)


if __name__ == "__main__":
    main()
