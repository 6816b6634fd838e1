#!/usr/bin/env python
"""bench.py -- descriptor-pairs/sec of the feature-matching path on N B200s (one process per GPU).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c3|c4|c5|c6]   # this repo's CUDA path
  python bench.py --impl reference [--gpus N] [--steps K] ...                       # the reference's CPU arithmetic

A "step" is one pass of the hot path over one synthetic descriptor set (BASELINE.json `configs`):
  global float (c2, c3, c6): K1 normalise/convert -> K2 tcgen05 candidates -> K3 exact re-rank -> K5 ratio filter +
                             compaction into match lists            (PP/featureMatching/featureMatchingGlobal.m:70-161)
  global binary (c4)        : K4 Hamming kNN -> K5                                   (PP/mex/flann_knn.cpp:199-223)
  pairwise (c5)             : per image pair 2-NN + ratio/threshold + unique         (featureMatchingPairwise.m:43-63)
Default workload: N=1 -> c2 = configs[1] (20 x 8192 SIFT-128, the configuration the metric is quoted on);
                  N>1 -> c3 = configs[2] (100 x 10000 SIFT-128 "sharded over 8 B200"): STRONG scaling of a fixed set --
                         query rows are sharded across ranks, every rank holds all train descriptors, the per-query
                         match records are exchanged with ONE NCCL all-gather and compacted.
`value`  : ordered descriptor pairs / device time of the step, inputs resident in HBM (max over ranks).
`e2e`    : same metric through the public call with pinned HOST buffers (H2D + D2H inside the timed region).
Prints ONE JSON line on rank 0.
--dump-outputs DIR: the match lists of the last timed step as DIR/<name>.npy (float64), for comparing two builds output
                    for output: pair_ptr [n*n + 1] (rows of cell (i, j) are pair_ptr[i + j*n] : pair_ptr[i + j*n + 1]),
                    matches [M x 2] (1-based feature indices, as in the `matches` cell) and, pairwise, metric [M].
"""
from __future__ import annotations

import os
import sys

if "--impl" in sys.argv and "reference" in sys.argv:
    # the CPU arm uses every host core even when the launcher (torch.distributed.run) exported OMP_NUM_THREADS=1;
    # must happen before numpy / OpenMP runtimes load
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(os.cpu_count() or 1)

import argparse  # noqa: E402
import json  # noqa: E402
import statistics  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "descriptor_pairs_per_sec"
UNIT = "pairs/s"
KNN = 4
CONFIGS = {   # name -> (synth config id, kind, workload label)
    "c2": (2, "global_float", "C2: 20 images x 8192 SIFT-128 f32 keypoints, global exhaustive k=4, ratio 0.8"),
    "c3": (3, "global_float", "C3: 100 images x 10000 SIFT-128 f32 keypoints, global exhaustive k=4, ratio 0.8"),
    "c6": (6, "global_float", "C2f: 20 images x 8192 REAL-valued SIFT-128 f32 keypoints, global exhaustive k=4, ratio 0.8"),
    "c4": (4, "global_binary", "C4: 50 images x 20000 ORB 256-bit keypoints, global BF Hamming k=4, ratio 0.8"),
    "c5": (5, "pairwise", "C5: 300 images x 4096 KAZE-64 f32 keypoints, pairwise exhaustive 2-NN, ratio 0.7, threshold 1.5"),
}
C5_INPUT = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.7, "useMATLABFeatureMatch": 0}
DUMP_LIMIT = 64 << 20   # bytes --dump-outputs may write; the largest, c5 (0.65 M match rows and their metric), needs about 16 MB


def default_config(n_gpus):
    return "c2" if n_gpus <= 1 else "c3"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"burst": d.get("bf16_tflops"), "sustained": d.get("bf16_tflops_sustained"), "hbm": d.get("hbm_gbs"),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6550.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = sorted(sm)[len(sm) // 2:] if sm else []  # upper half of the samples = under load
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- CPU arms (the only places that execute oracle/) -------------------------------------------------------------
def _oracle_all_cores():
    from oracle import oracle

    oracle.build(ref=False)
    oracle.set_num_threads(os.cpu_count() or 1)
    return oracle


def cpu_sample_global(oracle, desc, kind, nq, q0=0):
    """Exact kNN (+ nothing else) of `nq` query rows against the full pooled set -- the O(F^2 D) part of one step."""
    if kind == "global_binary":
        X = np.ascontiguousarray(np.concatenate(desc))
        t0 = time.perf_counter()
        idx, dist = oracle.knn_hamming(X, X[q0:q0 + nq], KNN)
    else:
        X = cpu_sample_global.cache.get(id(desc))
        if X is None:
            X = oracle.normalize_rows_global(np.concatenate(desc))
            cpu_sample_global.cache = {id(desc): X}
        t0 = time.perf_counter()
        idx, dist = oracle.knn_l2(X, X[q0:q0 + nq], KNN)
    return time.perf_counter() - t0, idx, dist, X


cpu_sample_global.cache = {}


def cpu_sample_pairwise(oracle, desc, npairs, first=0):
    """matchFeaturesScratch ('Exhaustive', Unique) of `npairs` image pairs of the column-major pair list."""
    n = len(desc)
    pl = [(i, j) for j in range(n) for i in range(j)]
    sel = [pl[(first + t * 977) % len(pl)] for t in range(npairs)]
    pairs = float(sum(desc[i].shape[0] * desc[j].shape[0] for i, j in sel))
    t0 = time.perf_counter()
    out = [oracle.match_features(desc[i], desc[j], C5_INPUT["Matchingthreshold"], C5_INPUT["Ratiothreshold"], True)
           for i, j in sel]
    return time.perf_counter() - t0, pairs, sel, out


def flann_kdtree_rate(X, exact_idx1, q0, nq):
    """The reference's DEFAULT global float engine (PP/mex/flann_knn.cpp:229-234: cv::flann::Index, KDTree(4),
    knnSearch(checks=32)) through the OpenCV python module of this image -- approximate and randomised, so it is
    reported beside the exact arm, never as the parity oracle.  Returns None when cv2 is not importable."""
    try:
        import cv2
    except Exception:
        return None
    cv2.setNumThreads(os.cpu_count() or 1)
    F = X.shape[0]
    t0 = time.perf_counter()
    index = cv2.flann_Index(X, dict(algorithm=1, trees=4))
    t_build = time.perf_counter() - t0
    t0 = time.perf_counter()
    idx, _ = index.knnSearch(X[q0:q0 + nq], KNN, params=dict(checks=32))
    t_search = time.perf_counter() - t0
    hits = sum(len(set(idx[r].tolist()) & set((exact_idx1[r] - 1).tolist())) for r in range(nq))
    total_s = t_build + t_search * F / nq
    return {"engine": f"cv2 {cv2.__version__} flann_Index KDTree(trees=4), knnSearch(checks=32); reference pins OpenCV 4.12",
            "value": F * float(F) / total_s, "unit": UNIT + " (F^2 / time: pair-equivalents of an approximate search)",
            "cores": 1, "build_s": t_build, "search_s_scaled": t_search * F / nq,
            "recall_at_k_vs_exact": hits / float(nq * KNN),
            "sample": f"index over all {F} rows, {nq} queries searched, search time scaled linearly"}


def blas_exhaustive_rate(X, nq):
    """The reference's own EXHAUSTIVE float arithmetic (PP/featureMatching/matchFeaturesScratch.m:343-358,
    nearest2SSDExhaustive: blocks of floor(1e7/N2) query rows, a2 + b2' - 2*A*B' by sgemm, min / mask / min) restated
    with numpy on this box's BLAS threads -- MATLAB would run the same three steps on MKL.  Extended here to the k = 4
    smallest per row (argpartition) so that it does the work of one global step.  Not bit-compatible with the oracle
    (sgemm summation order), so it is a timing arm only."""
    F = X.shape[0]
    block = max(1, int(1e7 // max(F, 1)))
    b2 = np.sum(X * X, axis=1, dtype=np.float32)
    t0 = time.perf_counter()
    for s0 in range(0, nq, block):
        A = X[s0:min(nq, s0 + block)]
        a2 = np.sum(A * A, axis=1, dtype=np.float32)
        D2 = (a2[:, None] + b2[None, :]) - np.float32(2) * (A @ X.T)
        part = np.argpartition(D2, KNN, axis=1)[:, :KNN]
        np.take_along_axis(D2, part, axis=1).sort(axis=1)
    dt = time.perf_counter() - t0
    return {"engine": "numpy sgemm + argpartition (nearest2SSDExhaustive's blocked GEMM form, k = %d)" % KNN,
            "value": nq * float(F) / dt, "unit": UNIT, "cores": os.cpu_count(),
            "sample": f"{nq} query rows x all {F} train rows in blocks of {block} rows ({dt:.1f} s), scaled linearly"}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: each array as out_dir/<name>.npy in float64 (exact for every index, offset and distance here)."""
    arrays = {name: np.ascontiguousarray(a, dtype=np.float64) for name, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"bench.py: the outputs take {total} bytes, more than --dump-outputs writes ({DUMP_LIMIT})")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def pairwise_csr_of_shares(counts, rows_all, met_all):
    """One CSR (pair_ptr, rows, metric) of the whole pair list from the per-rank shares in the layout of
    multigpu.exchange_pairwise_lists (counts [world x cells], rows [world x Mmax x 2], metric [world x Mmax]); every cell
    was computed by exactly one rank."""
    starts = np.cumsum(counts, axis=1) - counts          # offset of each cell in its rank's buffer
    total = counts.sum(axis=0)
    owner = counts.argmax(axis=0)
    spans = [(owner[c], starts[owner[c], c], starts[owner[c], c] + total[c]) for c in np.flatnonzero(total)]
    rows = np.concatenate([rows_all[r, a:b] for r, a, b in spans] or [np.zeros((0, 2), rows_all.dtype)])
    met = np.concatenate([met_all[r, a:b] for r, a, b in spans] or [np.zeros(0, met_all.dtype)])
    return np.concatenate([[0], np.cumsum(total)]), rows, met


def base_config(cfg, desc, ratio):
    """The `config` object: identical keys and values on both arms."""
    label = CONFIGS[cfg][2]
    F = int(sum(d.shape[0] for d in desc))
    if CONFIGS[cfg][1] == "pairwise":
        pairs = float(sum(desc[i].shape[0] * desc[j].shape[0] for j in range(len(desc)) for i in range(j)))
    else:
        pairs = float(F) * float(F)
    return {"workload": label, "F": F, "k": KNN if CONFIGS[cfg][1] != "pairwise" else 2, "ratio": ratio,
            "pairs_per_step": pairs}


def run_reference(args, rank, world):
    """--impl reference: the reference path's own CPU arithmetic on this box's host cores.
    MATLAB cannot run here and flann_knn.cpp needs OpenCV C++ (absent), so this is the oracle port (exact search
    with FLANN's own L2 functor, bit-identical distances to OpenCV's; BFMatcher-equivalent Hamming; the
    matchFeaturesScratch exhaustive branch) with all OpenMP threads, each step a bounded sample of the workload."""
    if rank != 0:
        return
    pkg = __import__("__graft_entry__").load_package()
    oracle = _oracle_all_cores()
    cfg = args.config or default_config(args.gpus)
    cid, kind, _ = CONFIGS[cfg]
    desc, c = pkg.synth.make_config(cid)
    ratio = C5_INPUT["Ratiothreshold"] if kind == "pairwise" else c["ratio"]
    config = base_config(cfg, desc, ratio)
    F = config["F"]
    budget = 150.0 / max(1, args.steps + args.warmup)      # whole run within a few minutes
    times, extra = [], {}
    if kind == "pairwise":
        dt, pairs, _, _ = cpu_sample_pairwise(oracle, desc, 1)
        npairs = int(max(1, min(64, min(3.0, budget) / max(dt, 1e-6))))
        for it in range(args.warmup + args.steps):
            dt, pairs, _, _ = cpu_sample_pairwise(oracle, desc, npairs, first=it * npairs)
            if it >= args.warmup:
                times.append(dt)
        unit_pairs = pairs
        sample = (f"{npairs} image pairs ({pairs:.3e} descriptor pairs) per step: exhaustive SSD 2-NN + ratio / threshold "
                  f"+ unique of the oracle, scaled linearly")
    else:
        cal = 256
        dt, _, _, X = cpu_sample_global(oracle, desc, kind, cal)
        rate = cal * F / dt
        nq = int(min(F, max(cal, rate * min(3.0, budget) / F)))
        for it in range(args.warmup + args.steps):
            q0 = (it * nq) % max(1, F - nq)
            dt, idx, dist, X = cpu_sample_global(oracle, desc, kind, nq, q0)
            if it >= args.warmup:
                times.append(dt)
        unit_pairs = float(nq) * F
        what = "exact Hamming kNN (BFMatcher order)" if kind == "global_binary" else "exact kNN, FLANN L2 functor order"
        sample = f"{nq} query rows x all {F} train rows per step ({what}, k={KNN}), scaled linearly"
        if kind == "global_float":
            approx = flann_kdtree_rate(X, idx, q0, nq)   # idx: the exact neighbours of the last timed sample
            if approx is not None:
                extra["reference_default_engine"] = approx
            extra["reference_exhaustive_blas"] = blas_exhaustive_rate(X, min(F, 4 * nq))
    ms = 1e3 * sum(times) / len(times)
    value = unit_pairs / (ms / 1e3)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None,
            "dtype": "u8" if kind == "global_binary" else "f32", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": oracle.num_threads(), "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    line.update(extra)
    print(json.dumps(line), flush=True)


# ---- this repo's CUDA path ---------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = __import__("__graft_entry__").load_package()
    L = pkg._lib.lib()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = pkg.Context(local_rank, stream=stream.cuda_stream)
    ctx.enable_timing(True)
    cfg = args.config or default_config(world)
    cid, kind, _ = CONFIGS[cfg]
    if kind == "pairwise":
        return run_ours_pairwise(args, rank, world, local_rank, pkg, ctx, stream, cfg, torch, dist)

    desc, c = pkg.synth.make_config(cid)   # same seed on every rank
    ratio = c["ratio"]
    config = base_config(cfg, desc, ratio)
    counts = [d.shape[0] for d in desc]
    n_img, F, D = len(desc), config["F"], desc[0].shape[1]
    is_binary = kind == "global_binary"
    pairs_total = config["pairs_per_step"]
    mg = pkg.multigpu

    # pinned host copies (what a MEX gateway hands over), row-major
    import ctypes as C
    host_ptrs, host_views = [], []
    for d in desc:
        p = L.aps_host_alloc(max(d.nbytes, 1))
        v = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_ubyte if is_binary else C.c_float)), shape=d.shape)
        v[...] = d
        host_ptrs.append(p)
        host_views.append(v)

    plan = pkg.GlobalPlan(ctx, counts, D, is_binary, KNN)
    plan.upload_pointers(host_ptrs)
    q0, q1 = mg.shard_bounds(F, world)[rank]
    rec = desc_dev = None
    if world > 1:
        rec = torch.as_tensor(mg.CudaView(plan.records_device(), (F + pkg.RECORD_PAD, 2), "<i4"), device="cuda")
        desc_dev = torch.as_tensor(mg.CudaView(plan.desc_device(), (F, D), "|u1" if is_binary else "<f4"), device="cuda")

    knn_ev = []

    def step_device(timed=False):
        plan.prepare()
        if timed:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
        plan.knn(q0, q1)
        if timed:
            e1.record(stream)
            knn_ev.append((e0, e1))
        plan.filter(ratio, q0, q1)
        if world > 1:
            mg.exchange_records(rec, F, world, rank, dist)
        plan.compact()

    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_device()
    barrier()
    ctx.tc_time()                                     # reset kernel-time accumulator
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.aps_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for s0, s1 in ev:
        flush.zero_()
        barrier()
        s0.record(stream)
        step_device(timed=True)
        s1.record(stream)
        barrier()
    launches = L.aps_launch_count() - launches0
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    knn_ms = sum(a.elapsed_time(b) for a, b in knn_ev) / max(1, len(knn_ev))
    tc_ms, tc_launches = ctx.tc_time()
    stats = ctx.last_stats()
    if world > 1:
        t = torch.tensor([total_ms, tc_ms, knn_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, tc_ms_max, knn_ms = float(t[0]), float(t[1]), float(t[2])
    else:
        tc_ms_max = tc_ms
    ms_per_step = total_ms / args.steps
    value = pairs_total / (ms_per_step / 1e3)
    multi_csr = plan.download() if rank == 0 else None     # the lists of the last timed step (all ranks' records)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pair_ptr": multi_csr[2], "matches": multi_csr[3]})

    # ---- end to end: pinned host buffers in, host match lists out -------------------------------
    def step_e2e():
        if world == 1:
            cells = [pkg.binaryFeatures(v) for v in host_views] if is_binary else host_views
            return pkg.featureMatchingGlobal({"k": KNN, "Ratiothreshold": ratio, "BFMatch": 1}, cells, n_img, ctx=ctx)
        # every rank uploads its own block of rows from pinned memory (all PCIe links in parallel), the blocks
        # are all-gathered over NVLink into the plan's pooled matrix
        mg.gather_descriptors(desc_dev, host_views, rank, world, dist, torch)
        step_device()
        return plan.download() if rank == 0 else None

    for _ in range(min(2, args.warmup)):
        step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = step_e2e()
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    clocks = sampler.stop() if rank == 0 else None

    if rank == 0:
        if world == 1:
            m_rows = sum(int(out[i][j].shape[0]) for j in range(n_img) for i in range(j) if out[i][j].ndim == 2)
        else:
            m_rows = int(out[3].shape[0])
        peaks = measured_peaks()
        details = {"l2": "512 MB buffer written between timed steps (L2 flush)",
                   "sharding": (f"query rows in {world} contiguous equal blocks; per-query records exchanged by ONE NCCL "
                                f"all-gather; e2e: every rank uploads its row block, NCCL all-gather of the blocks")
                   if world > 1 else "single GPU",
                   "engine": stats["engine"] if not is_binary else "hamming (CUDA cores, POPC)",
                   "fallback_rows_last_step": stats["fallback_rows"], "first_proof_unproven_rows": ctx.first_pass_unproven(),
                   "operands_exact_in_fp16": stats["bf16_exact_operands"],
                   "match_rows": m_rows, "knn_stage_ms": knn_ms}
        if is_binary:
            # dominant kernel: k_knn_hamming (the whole kNN stage is that one launch).  Algorithmic bytes per pair = the
            # train descriptor's nb operand bytes (SURVEY 8(d)); operands are re-used from shared memory, so the
            # HBM-equivalent figure may exceed 1.0 -- the true ceiling is the POPC issue rate.
            achieved = float(q1 - q0) * float(F) * D / (knn_ms / 1e3) / 1e9
            roof = {"bound": "hbm", "kernel": "k_knn_hamming", "achieved": achieved, "peak": peaks["hbm"], "unit": "GB/s",
                    "frac": achieved / peaks["hbm"], "peak_kind": f"HBM copy bandwidth, {peaks['source']}",
                    "kernel_ms": knn_ms, "kernel_share_of_step": knn_ms / ms_per_step, "traffic": None,
                    "note": "operand-stream equivalent (pairs x 32 B / time); POPC-pipe bound, see profiles/"}
            dtype = "u8"
        else:
            details["arithmetic"] = "fp16 tcgen05 operands (kind::f16), f32 accumulate, exact f32 re-rank of the candidates"
            # dominant kernel: k_knn_tc.  Algorithmic FLOPs per launch = 2*D * (rows of this rank) * F
            flops_per_launch = 2.0 * D * float(q1 - q0) * float(F)
            tc_avg_ms = tc_ms_max / max(1, args.steps)       # all tensor launches of one step (first + second pass)
            achieved = flops_per_launch / (tc_avg_ms / 1e3) / 1e12
            traffic = None
            tp = os.path.join(ROOT, "profiles", "traffic.json")
            if os.path.exists(tp) and world == 1 and cfg == "c2":   # ncu --set full on exactly this workload (profiles/)
                traffic = json.load(open(tp)).get("k_knn_tc_dram_bytes_per_launch")
            # a 6 ms step inside a 0.1 s timed region is burst-class (clocks at max, no power cap): burst peak
            roof = {"bound": "tensor", "kernel": "k_knn_tc", "achieved": achieved, "peak": peaks["burst"],
                    "unit": "TFLOP/s", "frac": achieved / peaks["burst"], "peak_kind": f"bf16 dense burst, {peaks['source']}",
                    "frac_of_sustained": achieved / peaks["sustained"], "kernel_ms": tc_avg_ms,
                    "tensor_launches_per_step": tc_launches / max(1, args.steps),
                    "kernel_share_of_step": tc_avg_ms / ms_per_step, "traffic": traffic}
            dtype = "f16"
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak",
            "vs_baseline": None, "dtype": dtype, "data": "synthetic", "config": config, "details": details,
            "roofline": roof,
            "e2e": {"value": pairs_total / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                    "h2d_bytes_per_step": F * D * (1 if is_binary else 4),
                    "d2h_bytes_per_step": (n_img * n_img + 1) * 8 + m_rows * 8},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if world > 1:
            # parity on the real NCCL path: the multi-rank CSR must equal a single-rank run of the same plan
            plan.prepare()
            plan.knn(0, F)
            plan.filter(ratio, 0, F)
            plan.compact()
            single = plan.download()
            same = (np.array_equal(single[2], multi_csr[2]) and np.array_equal(single[3], multi_csr[3]))
            line["parity_check"] = ("ok" if same else "MISMATCH") + (f": {world}-rank CSR (pair_ptr, {multi_csr[3].shape[0]} "
                                                                     f"rows) == 1-rank CSR of the same plan, bit for bit")
            rp = os.path.join(ROOT, "profiles", f"r2_bench_{cfg}_1gpu.json")
            if os.path.exists(rp):   # strong-scaling context: this workload on ONE GPU (recorded run of this bench)
                one = json.load(open(rp))
                line["strong_scaling"] = {"one_gpu_ms_per_step_recorded": one["ms_per_step"],
                                          "speedup": one["ms_per_step"] / ms_per_step,
                                          "source": f"profiles/r2_bench_{cfg}_1gpu.json"}
        if world == 1 and not args.no_cpu_baseline:
            oracle = _oracle_all_cores()
            cal = 256
            dt, _, _, _ = cpu_sample_global(oracle, desc, kind, cal)
            nq = int(min(F, max(cal, cal * 12.0 / dt)))
            dt, oi, od, _ = cpu_sample_global(oracle, desc, kind, nq)
            line["cpu_baseline"] = {"value": nq * float(F) / dt, "unit": UNIT, "cores": oracle.num_threads(), "kind": "port",
                                    "sample": f"{nq} query rows x all {F} train rows ({dt:.1f} s, exact kNN k={KNN} of the "
                                              f"oracle, scaled linearly)"}
            gi, gd = plan.download_knn(0, nq)   # the kNN table of the last step against the sample the CPU just searched
            same = np.array_equal(gi, oi) and np.array_equal(gd.view(np.uint32), od.view(np.uint32))
            line["parity_check"] = ("ok" if same else "MISMATCH") + f": kNN rows [0,{nq}) == oracle (indices and float bits)"
        if world == 1 and cfg == "c2" and not args.no_extra:
            line["config6_real_valued_ms"] = real_valued_step_ms(pkg, ctx, torch, stream, flush, args.steps)
        print(json.dumps(line), flush=True)
    plan.close()
    for p in host_ptrs:
        L.aps_host_free(p)
    if world > 1:
        dist.destroy_process_group()


def real_valued_step_ms(pkg, ctx, torch, stream, flush, steps):
    """The C2-sized set with REAL-valued SIFT-like descriptors (synth config 6: not exactly representable in bf16, what
    MATLAB's single SIFT / KAZE deliver): device ms per step of the same pipeline, beside the integer-SIFT headline."""
    desc, c = pkg.synth.make_config(6)
    plan = pkg.GlobalPlan(ctx, [d.shape[0] for d in desc], desc[0].shape[1], False, KNN)
    plan.upload(desc)

    def step():
        plan.prepare()
        plan.knn(0, plan.F)
        plan.filter(c["ratio"], 0, plan.F)
        plan.compact()

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    ms = []
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step()
        e1.record(stream)
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    st = ctx.last_stats()
    first = ctx.first_pass_unproven()
    plan.close()
    return {"ms_per_step": sum(ms) / len(ms), "fallback_rows": st["fallback_rows"], "engine": st["engine"],
            "first_proof_unproven_rows": first, "first_proof_unproven_frac": first / float(plan.F),
            "workload": CONFIGS["c6"][2]}


def run_ours_pairwise(args, rank, world, local_rank, pkg, ctx, stream, cfg, torch, dist):
    """c5: the pairwise sweep; image pairs of the column-major pair list are dealt block-cyclically to the ranks."""
    from importlib import import_module

    host = import_module(pkg.__name__ + ".host")
    L = pkg._lib.lib()
    cid = CONFIGS[cfg][0]
    desc, c = pkg.synth.make_config(cid)
    n = len(desc)
    config = base_config(cfg, desc, C5_INPUT["Ratiothreshold"])
    pairs_total = config["pairs_per_step"]
    inp = dict(C5_INPUT)
    F, D = config["F"], desc[0].shape[1]
    plan = pkg.PairwisePlan(ctx, [d.shape[0] for d in desc], D, False)
    plan.upload(desc)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def step_device():
        plan.prepare()
        return plan.match(inp["Matchingthreshold"], inp["Ratiothreshold"], rank, world)   # CSR of this rank's share (host)

    for _ in range(args.warmup):
        step_device()
    barrier()
    ctx.tc_time()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = L.aps_launch_count()
    times = []
    for _ in range(args.steps):
        flush.zero_()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        mine = step_device()
        e1.record(stream)
        barrier()
        times.append(e0.elapsed_time(e1))
    launches = L.aps_launch_count() - launches0
    tc_ms, tc_launches = ctx.tc_time()
    stats = ctx.last_stats()
    if args.dump_outputs:   # every rank's share of the last timed step, merged on rank 0
        shares = ((np.diff(mine[0])[None], mine[1][None], mine[2][None]) if world == 1 else
                  pkg.multigpu.exchange_pairwise_lists(*mine, world, dist, torch, "cuda"))
        if rank == 0:
            pp, rows, met = pairwise_csr_of_shares(*shares)
            dump_outputs(args.dump_outputs, {"pair_ptr": pp, "matches": rows, "metric": met})
    total_ms = sum(times)
    if world > 1:
        t = torch.tensor([total_ms, tc_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, tc_ms = float(t[0]), float(t[1])
    ms_per_step = total_ms / args.steps
    value = pairs_total / (ms_per_step / 1e3)

    # pinned host copies of the descriptor matrices (what a MEX gateway would stage), one per image
    import ctypes as C
    host_ptrs, host_views = [], []
    for d in desc:
        p = L.aps_host_alloc(max(d.nbytes, 1))
        v = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_float)), shape=d.shape)
        v[...] = d
        host_ptrs.append(p)
        host_views.append(v)
    desc_dev = torch.as_tensor(pkg.multigpu.CudaView(plan.desc_device(), (F, D), "<f4"), device="cuda")

    def step_e2e():
        """Pinned host descriptors in -> compacted match lists (CSR: per-cell counts, rows, metric) on the host of
        EVERY rank.  Each rank uploads its block of rows (all PCIe links in parallel), the blocks are all-gathered
        over NVLink, each rank matches its share of the pair list, counts-then-lists NCCL all-gather of the lists."""
        pkg.multigpu.gather_descriptors(desc_dev, host_views, rank, world, dist, torch)
        plan.prepare()
        pp, rows, met = plan.match(inp["Matchingthreshold"], inp["Ratiothreshold"], rank, world)
        if world == 1:
            return np.diff(pp)[None, :], rows[None, :, :], met[None, :]
        return pkg.multigpu.exchange_pairwise_lists(pp, rows, met, world, dist, torch, "cuda")

    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        csr = step_e2e()
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t[0])
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        peaks = measured_peaks()
        cells = pkg.merge_pairwise_csr(n, *csr)      # the n x n cell of featureMatchingPairwise (outside the timed region)
        m_rows = int(sum(cells[i][j].shape[0] for j in range(n) for i in range(j)))
        my_pairs = pairs_total / world
        tc_avg_ms = tc_ms / max(1, args.steps)
        achieved = 2.0 * D * my_pairs / (tc_avg_ms / 1e3) / 1e12
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
                "config": config,
                "details": {"engine": stats["engine"], "pairwise_stats": ctx.pairwise_stats(),
                            "arithmetic": "fp16 tcgen05 operands; screen: f16 accumulate (error-bounded rejection); "
                                          "surviving pairs: f32 accumulate + exact f32 re-rank of the candidates", "fallback_rows_last_step": stats["fallback_rows"],
                            "match_rows": m_rows, "image_pairs": n * (n - 1) // 2,
                            "sharding": f"image pairs dealt block-cyclically to {world} rank(s); counts-then-lists NCCL "
                                        f"all-gather of the compacted lists" if world > 1 else "single GPU",
                            "e2e_result": "compacted match lists (per-cell counts, [M x 2] rows, metric) on the host of every rank",
                            "l2": "512 MB buffer written between timed steps (L2 flush)"},
                "roofline": {"bound": "tensor", "kernel": "k_pair_screen (fp16 tcgen05 screen of all pairs) + k_knn_tc (exact stage on the surviving pairs)", "achieved": achieved,
                             "peak": peaks["burst"], "unit": "TFLOP/s", "frac": achieved / peaks["burst"],
                             "peak_kind": f"bf16 dense burst, {peaks['source']}", "kernel_ms": tc_avg_ms,
                             "tensor_launches_per_step": tc_launches / max(1, args.steps),
                             "kernel_share_of_step": tc_avg_ms / ms_per_step, "traffic": None},
                "e2e": {"value": pairs_total / e2e_s, "unit": UNIT, "ms_per_step": e2e_s * 1e3,
                        "h2d_bytes_per_step": F * D * 4, "d2h_bytes_per_step": (n * n + 1) * 8 + m_rows * 16},
                "gpu_launches": int(launches), "clocks": clocks}
        if not args.no_cpu_baseline:
            oracle = _oracle_all_cores()
            dt, pairs, sel, ref = cpu_sample_pairwise(oracle, desc, 24)
            if world == 1:
                line["cpu_baseline"] = {"value": pairs / dt, "unit": UNIT, "cores": oracle.num_threads(), "kind": "port",
                                        "sample": f"{len(sel)} image pairs ({pairs:.3e} descriptor pairs, {dt:.1f} s): "
                                                  f"matchFeaturesScratch exhaustive + unique of the oracle, scaled linearly"}
            same = all(np.array_equal(cells[i][j], m.astype(np.float64)) for (i, j), (m, _) in zip(sel, ref))
            line["parity_check"] = ("ok" if same else "MISMATCH") + f": {len(sel)} sampled image pairs == oracle match lists"
        rp = os.path.join(ROOT, "profiles", f"r2_bench_{cfg}_1gpu.json")
        if world > 1 and os.path.exists(rp):   # strong-scaling context: this workload on ONE GPU (recorded run of this bench)
            one = json.load(open(rp))
            line["strong_scaling"] = {"one_gpu_ms_per_step_recorded": one["ms_per_step"],
                                      "speedup": one["ms_per_step"] / ms_per_step,
                                      "source": f"profiles/r2_bench_{cfg}_1gpu.json"}
        print(json.dumps(line), flush=True)
    plan.close()
    for p in host_ptrs:
        L.aps_host_free(p)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps of every timed loop (at least 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=None, choices=sorted(CONFIGS), help="default: c2 on one GPU, c3 on several")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the real-valued (config 6) side measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the match lists of the last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(3, args.warmup)   # timing rule: at least 3 untimed warm-up steps
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        if world != args.gpus and world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
