"""CPU emulation (numpy, no GPU) of the two candidate epilogues of the batched pairwise tensor pass and of the
re-rank's rejection / completeness tests, to predict which share of the rows reaches the exact fallback.
usage: python profiles/emulate_pairwise_proofs.py [cid=5] [kp=4096] [ratio=0.7] [match_threshold=1.5]

  streaming : one top-4 list per (query, train image); proven iff  s~(4th) - eps > d2
  segment   : two lists (even / odd 64-column segments) of the three best of "two best per segment"; a column outside a
              list is bounded by the list's third entry; when a list's two best share a segment that segment is scanned
              exactly (emulated as: it never fails the proof by itself)
  rejected  : m1 - eps > ratio^2 (m2 + eps)  or  m1 - eps > match_threshold   (no exact distance needed)
bf16 operands are emulated by rounding the descriptors to bf16 (torch), eps as in csrc/aps_exact_math.cuh."""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as ge  # noqa: E402

pkg = ge.load_package()
cid = int(sys.argv[1]) if len(sys.argv) > 1 else 5
kp = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
ratio = float(sys.argv[3]) if len(sys.argv) > 3 else 0.7
mt = float(sys.argv[4]) if len(sys.argv) > 4 else 1.5
desc, _ = pkg.synth.make_config(cid, n=4, kp=kp)
SEG = 64
SEG_LEN = int(os.environ.get("SEG_LEN", "3"))   # entries per segment list (round 1 ships 3; SEG_LEN=4: branch round2-wip)


def bf16(x):
    return torch.tensor(x).bfloat16().float().numpy()


def exact(A, B, idx):
    return np.stack([((A - B[idx[:, i]]) ** 2).sum(1) for i in range(idx.shape[1])], 1)


def run(A, B, label):
    if max(np.abs(A).max(), np.abs(B).max()) > 2:     # matchFeaturesScratch.m:105-110
        A = A / (np.sqrt((A * A).sum(1, keepdims=True)) + np.float32(1.1920929e-07))
        B = B / (np.sqrt((B * B).sum(1, keepdims=True)) + np.float32(1.1920929e-07))
    N, M = A.shape[0], B.shape[0] // SEG * SEG
    B = B[:M]
    sqA, sqB = (A * A).sum(1), (B * B).sum(1)
    score = bf16(A) @ bf16(B).T - 0.5 * sqB[None, :]
    maxsq = max(1.0, float(max(sqA.max(), sqB.max())))
    eps0 = (1e-4 + 1.57e-2) * maxsq
    r2 = ratio * ratio
    # streaming top-4
    o4 = np.argsort(-score, axis=1)[:, :4]
    s4 = sqA[:, None] - 2 * np.take_along_axis(score, o4, 1)
    e4 = np.sort(exact(A, B, o4), 1)
    rej4 = (s4[:, 0] - eps0 > r2 * (s4[:, 1] + eps0)) | (s4[:, 0] - eps0 > mt)
    unp4 = ~(s4[:, 3] - eps0 > e4[:, 1]) & ~rej4
    # segment epilogue
    eps1 = eps0 + 5e-5 * maxsq
    S = score.reshape(N, M // SEG, SEG)
    top = -np.sort(-S, axis=2)[:, :, :2]
    arg = np.argsort(-S, axis=2)[:, :, :2] + (np.arange(M // SEG) * SEG)[None, :, None]
    W = np.full(N, np.inf)
    idx, sap = [], []
    for ch in (0, 1):
        U, UI = top[:, ch::2, :].reshape(N, -1), arg[:, ch::2, :].reshape(N, -1)
        o = np.argsort(-U, axis=1)[:, :SEG_LEN]
        L, LI = np.take_along_axis(U, o, 1), np.take_along_axis(UI, o, 1)
        s = sqA[:, None] - 2 * L
        W = np.minimum(W, s[:, SEG_LEN - 1])
        idx.append(LI), sap.append(s)
    idx, sap = np.concatenate(idx, 1), np.concatenate(sap, 1)
    ss = np.sort(sap, 1)
    rej = (ss[:, 0] - eps1 > r2 * (ss[:, 1] + eps1)) | (ss[:, 0] - eps1 > mt)
    unp = ~(W - eps1 > np.sort(exact(A, B, idx), 1)[:, 1]) & ~rej
    print(f"{label}: rejected without exact distances {100 * rej4.mean():5.1f} % | to the exact fallback: streaming "
          f"{100 * unp4.mean():.2f} %, segment {100 * unp.mean():.2f} %")


run(desc[0], desc[1], "overlapping pair (30 % shared keypoints)")
run(desc[0], np.roll(desc[3], 1, axis=1), "unrelated pair (dimensions rotated)      ")
# r1 (C5 family, 4096 KAZE-64 keypoints per image, ratio 0.7, threshold 1.5):
#   overlapping pair: rejected 61.8 % | to the exact fallback: streaming 0.56 %, segment 1.39 % (SEG_LEN=3), 0.05 % (SEG_LEN=4)
#   unrelated pair  : rejected 100 %  | 0 / 0
# the segment lists lose when the three best columns overall fall into the same list (25 %): W is then the 3rd best overall
# instead of the 4th.  Four entries per list (W = min of the lists' 4th entries >= the 4th best overall) would close that gap.
