"""Device input against the host route for a caller whose descriptors and keypoints are already CUDA tensors, alternated
in one run:
  host route    the caller downloads the tensors (.cpu().numpy(), pageable) and calls globalImageMatchingSets /
                pairwiseImageMatchingSets, which upload them again;
  device route  globalImageMatchingSetsDevice / pairwiseImageMatchingSetsDevice on the tensors themselves.

    python profiles/time_device_inputs.py [reps]

Batches (make_set of tests/test_gpu_global_image_matching.py: SIFT-like 128-dimensional float32 descriptors on rings,
float64 keypoints; k 4 / Matchingthreshold 1.5, Ratiothreshold 0.8, Exhaustive, m = 6, maxIter 500, maxDistance 5.5,
confidence 99.9): config 2's shape as one set (20 x 8192), config 5's shape as one set (300 x 4096; SIFT-like rather
than KAZE-64) and as its 10 rings of 30 images, and 64 sets of 6 x 300.  Both routes end with every set's allMatches,
numMatches and tforms on the host.  Each repetition runs the two routes back to back (the order alternating); the times
are the median (min / max) of `reps` repetitions after one warm-up of each, host clock around calls that end in a
device synchronisation.  The outputs of both routes are compared bit for bit in the same run.  Prints the card, its
power limit and its maximum SM clock."""
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
from time_pairwise_image_matching import same  # noqa: E402

GLOBAL = {"k": 4, "Ratiothreshold": 0.8, "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500,
          "mBrownLowe": 6}
PAIRWISE = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.8, "useMATLABFeatureMatch": 0,
            "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}


def batch(aps, B, n, kp, seed):
    import torch

    rng = np.random.default_rng(seed)
    d, k = [], []
    for _ in range(B):
        cells, kps = make_set(aps, rng, n, kp)
        d.append([torch.from_numpy(np.asarray(c, np.float32)).cuda() for c in cells])
        k.append([torch.from_numpy(np.ascontiguousarray(x, np.float64)).cuda() for x in kps])
    return d, k, [n] * B


def main():
    import torch

    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
    print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    aps = ge.load_package()
    cases = [("1 x C2 (20 x 8192)", lambda: batch(aps, 1, 20, 8192, 100)),
             ("C5 (300 x 4096)", lambda: batch(aps, 1, 300, 4096, 250)),
             ("C5 as 10 rings", lambda: batch(aps, 10, 30, 4096, 200)),
             ("64 x (6 x 300)", lambda: batch(aps, 64, 6, 300, 300))]
    print(f"{'batch':>20} {'verb':>8} {'MB in':>7} {'host route ms':>24} {'device route ms':>24} {'saved':>6}  outputs",
          flush=True)
    for name, make in cases:
        d, k, ns = make()
        mb = sum(t.numel() * t.element_size() for s in d + k for t in s) / 1e6
        for verb, inp in (("global", GLOBAL), ("pairwise", PAIRWISE)):
            host = getattr(aps, f"{verb}ImageMatchingSets")
            dev = getattr(aps, f"{verb}ImageMatchingSetsDevice")

            def host_route():
                hd = [[t.cpu().numpy() for t in s] for s in d]
                hk = [[t.cpu().numpy() for t in s] for s in k]
                r = host(inp, hd, ns, hk)
                return r, host.last

            def dev_route():
                return dev(inp, d, ns, k), dev.last

            times = {"host": [], "dev": []}
            outs = {}
            for rep in range(reps + 1):
                for route in (("host", "dev") if rep % 2 == 0 else ("dev", "host")):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    outs[route] = (host_route if route == "host" else dev_route)()
                    dt = (time.perf_counter() - t0) * 1e3
                    if rep > 0:
                        times[route].append(dt)
            ok = same(outs["host"][0], outs["dev"][0], outs["host"][1], outs["dev"][1])
            h, v = np.median(times["host"]), np.median(times["dev"])
            fmt = lambda t: f"{np.median(t):8.2f} ({min(t):7.2f} / {max(t):7.2f})"   # noqa: E731
            print(f"{name:>20} {verb:>8} {mb:7.1f} {fmt(times['host']):>24} {fmt(times['dev']):>24} {h - v:6.1f}  "
                  f"{'identical' if ok else 'DIFFERENT'}", flush=True)


if __name__ == "__main__":
    main()
