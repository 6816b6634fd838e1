"""Inputs for the tensor kNN contract tests (tests/test_gpu_tc_contract.py, tests/test_tc_adversarial_data_cpu.py).

Adversarial rounding: the re-rank proves a row's top-k complete from approximate distances whose error it bounds by
eps_bound (csrc/aps_exact_math.cuh).  On random data the operand rounding errors partly cancel, so a bound several
times too small goes unnoticed.  Here every component of the query and of its true neighbours sits just below a
rounding midpoint of the 16-bit operand type and rounds toward zero, so the approximate distance of a true neighbour
is inflated by nearly the whole operand term.  A crowd of rows, exactly farther by a small gap, rounds the same way on
most components but away from zero on a few: it is inflated a little less, outranks the true neighbours in the
approximate order and fills the candidate lists.  Only a sound eps keeps such a row from being "proven" with the crowd.
"""
import numpy as np

D = 128
# operand-rounding term of eps_bound, per unit of max|x|^2: it must cover 2 (2u + u^2) |a||b|, u = unit roundoff
EPS_TERM = {"bf16": 1.57e-2, "fp16": 2.0e-3}
UNIT_ROUNDOFF = {"bf16": 2.0 ** -8, "fp16": 2.0 ** -11}
E32 = 2.0 ** -23  # float32 spacing in [1, 2)


def bf16_round(x):
    """float32 -> nearest-even bfloat16, returned as float32."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    r = ((u + 0x7FFF + ((u >> 16) & 1)) >> 16) << 16
    return r.astype(np.uint32).view(np.float32)


def round_operand(x, fmt):
    x = np.asarray(x, np.float32)
    return bf16_round(x) if fmt == "bf16" else x.astype(np.float16).astype(np.float32)


def inflation(q, T, fmt):
    """2 (q.t - q~.t~) per row of T, in float64: how much the operand rounding adds to the approximate distance."""
    q64, T64 = q.astype(np.float64), T.astype(np.float64)
    qr, Tr = round_operand(q, fmt).astype(np.float64), round_operand(T, fmt).astype(np.float64)
    return 2.0 * (T64 @ q64 - Tr @ qr)


def approx_l2(q, T, fmt):
    """|q|^2 + |t|^2 - 2 q~.t~ in float64: the distance the candidate kernel ranks by (before fp32 accumulation)."""
    q64, T64 = q.astype(np.float64), T.astype(np.float64)
    qr, Tr = round_operand(q, fmt).astype(np.float64), round_operand(T, fmt).astype(np.float64)
    return (q64 @ q64) + (T64 * T64).sum(1) - 2.0 * (Tr @ qr)


def exact_l2(q, T):
    d = T.astype(np.float64) - q.astype(np.float64)
    return (d * d).sum(1)


def planted_group(fmt, rng, n_true=4, n_crowd=128, n_up=12, n_shift=24, shift_cells=2):
    """One planted group: rows [0, n_true) = the query and its true neighbours, rows [n_true, n_true + n_crowd) = the
    crowd.  Components are +-(1 + u - a 2^-23) (a small: rounds toward zero); the sign pattern is random, so groups
    are far apart.  The true neighbours differ from the query by a few float32 ulps.  A crowd row moves n_shift
    components by shift_cells whole operand cells (same offset in the cell: still rounds toward zero; this sets the
    gap) and puts n_up others just above the midpoint (rounds away from zero: less inflation)."""
    u = UNIT_ROUNDOFF[fmt]
    sign = np.where(rng.random(D) < 0.5, -1.0, 1.0)
    mag = np.full(D, 1.0 + u - 4 * E32)
    rows = np.empty((n_true + n_crowd, D))
    rows[0] = mag
    for j in range(1, n_true):  # j components one ulp lower: exact distance j 2^-46, still below the midpoint
        t = mag.copy()
        t[rng.choice(D, j, replace=False)] -= E32
        rows[j] = t
    for c in range(n_crowd):
        t = mag.copy()
        pick = rng.choice(D, n_up + n_shift, replace=False)
        t[pick[:n_up]] = 1.0 + u + 4 * E32
        t[pick[n_up:]] += shift_cells * 2 * u
        rows[n_true + c] = t
    return (rows * sign).astype(np.float32)


def _far_groups_of_four(rng, n_groups, norm, clip=None):
    """Background: groups of four near-identical rows in random directions, far from each other and from the planted
    rows: every background row's top-4 is its group, with a gap far above eps (it is proven on the first pass)."""
    centers = rng.standard_normal((n_groups, D))
    centers *= norm / np.linalg.norm(centers, axis=1, keepdims=True)
    rows = np.repeat(centers, 4, axis=0) + 1e-3 * rng.standard_normal((4 * n_groups, D))
    if clip is not None:
        rows = np.clip(rows, -clip, clip)
    return rows.astype(np.float32)


def flann_adversarial_set(F=4096, n_groups=2, seed=0):
    """bf16 through flann_knn_win (raw rows, bias -|t|^2/2): X [F x D] and, per planted group, the row indices of its
    query + true neighbours and of its crowd.  The crowd rows are spread evenly over the rows, so that every column
    segment of the candidate kernel holds more of them than a list keeps."""
    rng = np.random.default_rng(seed)
    groups = [planted_group("bf16", rng) for _ in range(n_groups)]
    n_planted = sum(g.shape[0] for g in groups)
    n_bg = (F - n_planted) // 4
    bg = _far_groups_of_four(rng, n_bg, norm=8.0)
    X = np.empty((F, D), np.float32)
    X[n_planted + 4 * n_bg:] = 0  # (F - n_planted) % 4 rows left over: zero rows, far from everything planted
    pos = rng.permutation(F)
    planted_pos, cur = [], 0
    for g in groups:
        idx = pos[cur:cur + g.shape[0]]
        X[idx] = g
        planted_pos.append((idx[:4], idx[4:]))
        cur += g.shape[0]
    X[pos[cur:cur + bg.shape[0]]] = bg
    return X, planted_pos


def pairwise_adversarial_set(n1=1024, n2=1024, n_groups=4, seed=1):
    """fp16 through matchFeaturesScratch Exhaustive (|x| <= 2: raw fp16 operands).  A holds each group's query, B its
    ONE true neighbour (so the ratio test accepts the match) and its crowd.  Returns A, B, per group (row of A,
    row of B of the true neighbour, rows of B of the crowd)."""
    rng = np.random.default_rng(seed)
    groups = [planted_group("fp16", rng, n_true=2, n_crowd=48, n_shift=40, shift_cells=4) for _ in range(n_groups)]
    A = _far_groups_of_four(rng, n1 // 4, norm=6.0, clip=2.0)
    B = _far_groups_of_four(rng, n2 // 4, norm=6.0, clip=2.0)
    pa = rng.choice(n1, n_groups, replace=False)
    pb = rng.permutation(n2)
    planted, cur = [], 0
    for g, ra in zip(groups, pa):
        A[ra] = g[0]
        rb = pb[cur:cur + g.shape[0] - 1]
        B[rb] = g[1:]
        planted.append((ra, rb[0], rb[1:]))
        cur += g.shape[0] - 1
    return A, B, planted


def degenerate_set(F, rng):
    """Integer-valued rows with ties and degenerate scales: 3 all-zero rows, 200 copies of one row, 20 constant rows
    (each its own value), the rest random 0..255."""
    X = rng.integers(0, 256, (F, D)).astype(np.float32)
    pos = rng.permutation(F)
    X[pos[:3]] = 0
    X[pos[3:203]] = X[pos[203]]
    for i, r in enumerate(pos[204:224]):
        X[r] = float(i * 13 % 256)
    return X
