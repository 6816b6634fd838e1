"""Per-tile cycle accounting of the long-sweep k_knn_tc epilogue on C2 (20 x 8192 integer SIFT-128, global k = 4).

Builds the package of TREE with -DAPS_TC_TILE_CLOCKS into a scratch directory (never into TREE), runs the C2 global
kNN twice (the first run warms up) and reads back one record per (epilogue warp, tile) of the second run's first-pass
launch: clock() cycles of the acc_full wait, the scan and vote, the walk of the flagged groups without its insertions
(staging, TMEM re-reads, waits for the column constants), the insertions, and the whole tile; the union of flagged
groups and the number of re-read rounds.  Prints histograms of fast and flagged tile cycles, the share of each phase
and the mean union and rounds.

    python profiles/tile_clocks.py [--tree TREE] [--work DIR] [--patch FILE] [--label NAME]

TREE must have the -DAPS_TC_TILE_CLOCKS path (this commit or later).  --patch applies a patch to the scratch copy
before it is built: profiles/r5_walk_ldg_before.patch gives the kernel before the column constants were prefetched
(its flagged walk loads them from L2 in every round), which is how profiles/r5_tile_clocks_before.txt was taken.
--work reuses a scratch build (objects are rebuilt only when a source is newer).  Needs a B200.

The measured variant is not the default kernel: the clock reads and their bookkeeping take registers (ptxas: 8 B stack,
4 B spill stores, 12 B spill loads in the non-bias long-sweep instantiations, the C2 kernel included, outside the tile
loop; the default build has none), and it waits for every column constant of a round before the insertions start, so
that this wait is counted in the walk.  Read the split as where a tile's cycles go, not as the default kernel's times.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib.util
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "automaticpanoramicimagestitching-autopanostitch-matlab_b200"
PHASES = ("wait acc_full", "scan + vote", "walk (re-read, constants)", "insertions", "rest of the tile")


def load_scratch_package(tree, work, patch=None):
    """Copies TREE's package sources into WORK, applies PATCH there and builds them with the tile-clock flag."""
    pdir = os.path.join(work, PKG)
    os.makedirs(pdir, exist_ok=True)
    for name in os.listdir(os.path.join(tree, PKG)):
        src = os.path.join(tree, PKG, name)
        if name.endswith(".py"):
            shutil.copy2(src, pdir)
    shutil.copytree(os.path.join(tree, PKG, "csrc"), os.path.join(pdir, "csrc"), dirs_exist_ok=True)
    shutil.copytree(os.path.join(tree, "include"), os.path.join(work, "include"), dirs_exist_ok=True)
    if patch:
        subprocess.run(["patch", "-p1", "-s", "-d", work, "-i", os.path.abspath(patch)], check=True)
    spec = importlib.util.spec_from_file_location("apsmatch_tile_clocks", os.path.join(pdir, "__init__.py"),
                                                  submodule_search_locations=[pdir])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["apsmatch_tile_clocks"] = mod
    # _lib only builds on request: add the flag before build_library reads NVCC_FLAGS
    lib_spec = importlib.util.spec_from_file_location("apsmatch_tile_clocks._lib", os.path.join(pdir, "_lib.py"))
    lib_mod = importlib.util.module_from_spec(lib_spec)
    sys.modules["apsmatch_tile_clocks._lib"] = lib_mod
    lib_spec.loader.exec_module(lib_mod)
    if "-DAPS_TC_TILE_CLOCKS" not in lib_mod.NVCC_FLAGS:
        lib_mod.NVCC_FLAGS.append("-DAPS_TC_TILE_CLOCKS")
    lib_mod.build_library()
    spec.loader.exec_module(mod)
    return mod


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def histogram(x, edges):
    h, _ = np.histogram(x, bins=edges)
    out = []
    for i, n in enumerate(h):
        hi = "inf" if not np.isfinite(edges[i + 1]) else f"{int(edges[i + 1])}"
        out.append(f"  [{int(edges[i]):>6}, {hi:>6})  {n:>9}  {100.0 * n / max(1, len(x)):5.1f} %  " +
                   "#" * int(round(60.0 * n / max(1, len(x)))))
    return "\n".join(out)


def fmt(v, fn=np.mean, spec=".0f"):
    return format(fn(v), spec) if len(v) else "-"


def report(rec, label):
    wait, scan, walk, ins, total = (rec[:, i].astype(np.int64) for i in range(5))
    uni, rounds, flags = rec[:, 5], rec[:, 6], rec[:, 7]
    rest = total - wait - scan - walk - ins
    flagged = (flags & 1) != 0
    first = (flags & 4) != 0
    if not len(rec):
        print(f"== {label}: no tile records")
        return
    print(f"== {label}: {len(rec)} tile records (epilogue warp x tile), flagged {flagged.mean():.3f}, "
          f"partial {((flags & 2) != 0).mean():.4f}, first tile of a unit {first.mean():.4f}")
    busy = total - wait
    for name, m in (("fast", ~flagged), ("flagged", flagged)):
        if not m.any():
            print(f"-- {name} tiles: none")
            continue
        print(f"-- {name} tiles ({m.sum()}): cycles per tile mean {total[m].mean():.0f}, busy (without the acc_full "
              f"wait) mean {busy[m].mean():.0f} median {np.median(busy[m]):.0f} p90 {np.percentile(busy[m], 90):.0f}")
        edges = np.array([0, 100, 200, 300, 400, 600, 800, 1000, 1500, 2000, 3000, 4000, 6000, 10000, np.inf])
        print("   busy cycles histogram:")
        print(histogram(busy[m], edges))
    print("-- share of the epilogue warps' cycles per phase (all tiles | fast | flagged, flagged mean cycles):")
    parts = (wait, scan, walk, ins, rest)

    def share(v, m):
        return f"{100.0 * v[m].sum() / total[m].sum():5.1f} %" if total[m].sum() > 0 else "    - "

    for name, v in zip(PHASES, parts):
        print(f"   {name:<28} {share(v, np.ones_like(flagged))} | {share(v, ~flagged)} | {share(v, flagged)}, "
              f"{fmt(v[flagged]):>7}")
    nf = flagged & ~first
    print(f"-- flagged tiles (not first of a unit, {nf.sum()}): union mean {fmt(uni[nf], spec='.2f')} groups, rounds "
          f"mean {fmt(rounds[nf], spec='.2f')}; walk per round {walk[nf].sum() / max(1, rounds[nf].sum()):.0f} cycles, "
          f"insertions per round {ins[nf].sum() / max(1, rounds[nf].sum()):.0f} cycles")
    for r in range(1, 5):
        m = nf & (rounds == r)
        if m.any():
            print(f"   {r} round(s): {m.sum():>8} tiles, walk mean {walk[m].mean():6.0f}, insertions mean "
                  f"{ins[m].mean():6.0f}, busy mean {busy[m].mean():6.0f}")
    print(f"-- mean over all tiles: {fmt(total)} cycles per tile step, busy {fmt(busy)}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=ROOT, help="repository tree whose kernel is measured")
    ap.add_argument("--work", default=None, help="scratch build directory (default: a temporary one)")
    ap.add_argument("--patch", default=None, help="patch applied to the scratch copy before it is built")
    ap.add_argument("--label", default=None)
    a = ap.parse_args()
    work = a.work or tempfile.mkdtemp(prefix="aps_tile_clocks_")
    pkg = load_scratch_package(os.path.abspath(a.tree), os.path.abspath(work), a.patch)
    L = pkg._lib.lib()
    fn = getattr(L, "aps_debug_tile_clocks")
    fn.restype, fn.argtypes = C.c_int, [C.c_int, C.c_void_p, C.c_void_p]
    shape = np.zeros(4, np.uint32)
    pkg._lib.check(fn(2, shape.ctypes.data, None))
    ctas, warps, cap, words = (int(v) for v in shape)

    desc, c = pkg.synth.make_config(2)
    ctx = pkg._lib.default_context()
    plan = pkg.GlobalPlan(ctx, [d.shape[0] for d in desc], desc[0].shape[1], False, 4)
    plan.upload(desc)
    plan.prepare()
    plan.knn()
    ctx.synchronize()
    pkg._lib.check(fn(0, None, None))
    plan.prepare()
    plan.knn()
    ctx.synchronize()
    counts = np.zeros(ctas * warps, np.uint32)
    recs = np.zeros((ctas * warps, cap, words), np.uint32)
    pkg._lib.check(fn(1, counts.ctypes.data, recs.ctypes.data))
    rec = np.concatenate([recs[w, :counts[w]] for w in range(ctas * warps)])
    print("card (name, power limit, max SM clock, SM clock after the run):", card())
    print(f"tree: {os.path.abspath(a.tree)}; C2 F = {plan.F}; records per warp: max {counts.max()}, "
          f"warps with records {int((counts > 0).sum())} (capacity {cap})")
    report(rec, a.label or os.path.basename(os.path.abspath(a.tree)))


if __name__ == "__main__":
    main()
