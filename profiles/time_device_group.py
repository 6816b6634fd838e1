"""One-call device-group matching (aps_group_feature_matching_global / _pairwise) on 1, 2, 4 and 8 GPUs of one process,
fed from PAGEABLE, COLUMN-MAJOR numpy arrays -- what a MEX call hands over (mxGetData of the descriptor cells).

C3 (global, 100 x 10000 SIFT-128, F = 1e6) and C5 (pairwise, 300 x 4096 KAZE-64).  Per group size: median host-clock
time per call over --calls calls after one warm-up call (each call ends with its lists on the host), and member 0's
device-side stage times of the last call (CUDA events on its stream): upload of its share of the host data, peer
exchange of the descriptors, search, and (global) gather + compaction + download.  The slowest member's search is
printed too.  Lists are compared with the 1-GPU call bit for bit.
usage: time_device_group.py [--calls 5] [--sizes 1,2,4,8] [--configs 3,5]"""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402

pkg = ge.load_package()
L = pkg._lib.lib()


def run_call(group, cid, mats, cnt, n, D, c):
    ptrs = (C.c_void_p * n)(*[m.ctypes.data for m in mats])
    h = C.c_void_p()
    t0 = time.perf_counter()
    if cid == 3:
        rc = L.aps_group_feature_matching_global(group.handle, ptrs, cnt, n, D, 0, pkg._lib.APS_COL_MAJOR, c["k"],
                                                 c["ratio"], 0, C.byref(h))
    else:
        rc = L.aps_group_feature_matching_pairwise(group.handle, ptrs, cnt, n, D, 0, pkg._lib.APS_COL_MAJOR, 1.5,
                                                   c["ratio"], 0, 12000, 0, C.byref(h))
    ms = (time.perf_counter() - t0) * 1e3
    pkg._lib.check(rc)
    try:
        csr = pkg.host._csr_from_matchlist(h, n)
    finally:
        L.aps_matchlist_free(h)
    return ms, csr


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--sizes", default="1,2,4,8")
    ap.add_argument("--configs", default="3,5")
    a = ap.parse_args()
    import torch

    ndev = torch.cuda.device_count()
    if ndev == 0:
        raise SystemExit("no GPU: nothing to measure")
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    print("GPUs (index, name, power limit):")
    print(q.stdout.strip() or q.stderr.strip())
    print(f"{ndev} visible; calls per size = {a.calls} after 1 warm-up; input: pageable column-major numpy arrays")
    for cid in [int(x) for x in a.configs.split(",")]:
        desc, c = pkg.synth.make_config(cid)
        mats = [np.asfortranarray(d) for d in desc]          # MATLAB layout, ordinary (pageable) memory
        n, D = len(mats), mats[0].shape[1]
        cnt = (C.c_int64 * n)(*[m.shape[0] for m in mats])
        print(f"\n{c['name']}  (F = {sum(m.shape[0] for m in mats)}, {sum(m.nbytes for m in mats) / 2**20:.0f} MiB)")
        print(f"{'GPUs':>4} {'median ms':>10} {'min ms':>8} {'speed-up':>8} | member 0 stages (ms): {'upload':>7} "
              f"{'exchange':>8} {'search':>7} {'finish':>7} | max search | identical")
        ref, base = None, None
        for N in [int(x) for x in a.sizes.split(",")]:
            if N > ndev:
                print(f"{N:>4} not measured: only {ndev} GPUs visible")
                continue
            group = pkg.DeviceGroup(list(range(N)))
            run_call(group, cid, mats, cnt, n, D, c)                 # warm-up: module loads, pools, peer mappings
            times, csr = [], None
            for _ in range(a.calls):
                ms, csr = run_call(group, cid, mats, cnt, n, D, c)
                times.append(ms)
            st = [group.stage_times(i) for i in range(N)]
            med = statistics.median(times)
            if ref is None:
                ref, base = csr, med
            same = all(np.array_equal(x, y) for x, y in zip(csr, ref))
            s0 = st[0]
            stages = (f"{s0['upload']:7.2f} {s0['exchange']:8.2f} {s0['search']:7.2f} {s0['finish']:7.2f}" if N > 1
                      else f"{'(one-member group: single-context call, no stage events)':>33}")
            print(f"{N:>4} {med:10.2f} {min(times):8.2f} {base / med:8.2f} | {'':22}{stages} | "
                  f"{max(s['search'] for s in st):10.2f} | {same}")
            group.close()


if __name__ == "__main__":
    main()
