"""GPU: the candidate lists of the tensor kNN kernel (k_knn_tc) against the contract the re-rank's completeness proof
relies on, variant by variant and schedule by schedule, plus end-to-end bit-exactness where the long-sweep variants
run and inputs whose operand rounding all points one way (tests/tc_contract_data.py).

The contract (aps_rerank.cu): let W be the largest minimum retained score over the row's FULL lists; every train
column in none of the row's lists scores at most W, and every slot the re-rank reads was written by this launch."""
import numpy as np
import pytest

import tc_contract_data as tcd

pytestmark = pytest.mark.gpu

SENT = 0xA5A5A5A5
EMPTY = 0xFFFFFFFF
INFO = ("sm_count", "nslot", "rows_full", "exact", "operand_kind", "pre", "units_full", "tail_units", "tail_seg",
        "tail_balanced", "tiles_per_seg")


def sm_count(aps):
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def tc_candidates(aps, Q, T, prep, q0=0, q1=None, t0=0, t1=None, rows=None, natural=False):
    ctx = aps._lib.default_context()
    L = aps._lib.lib()
    T = np.ascontiguousarray(T, np.float32)
    Q = T if Q is None else np.ascontiguousarray(Q, np.float32)
    nq, nt, D = Q.shape[0], T.shape[0], T.shape[1]
    q1 = nq if q1 is None else q1
    t1 = nt if t1 is None else t1
    nr = q1 - q0
    cidx = np.zeros(nr * 32, np.uint32)
    csc = np.zeros(nr * 32, np.float32)
    perm = np.zeros(nt, np.int32)
    qb = np.zeros((nq, D), np.uint16)
    tb = np.zeros((nt, D), np.uint16)
    cs = np.zeros(nt, np.float32)
    cb = np.zeros(nt, np.float32)
    info = np.zeros(11, np.int64)
    r = None if rows is None else np.ascontiguousarray(rows, np.int32)
    aps._lib.check(L.aps_debug_tc_candidates(
        ctx.handle, Q.ctypes.data, nq, T.ctypes.data, nt, D, prep, int(natural), q0, q1, t0, t1,
        None if r is None else r.ctypes.data, 0 if r is None else len(r), cidx.ctypes.data, csc.ctypes.data,
        perm.ctypes.data, qb.ctypes.data, tb.ctypes.data, cs.ctypes.data, cb.ctypes.data, info.ctypes.data))
    inf = dict(zip(INFO, info.tolist()))
    ns = inf["nslot"]
    return dict(info=inf, cidx=cidx[:nr * ns * 8].reshape(nr, ns, 8), csc=csc[:nr * ns * 8].reshape(nr, ns, 8),
                perm=perm, qb=qb, tb=tb, colscale=cs, colbias=cb, q0=q0, q1=q1, t0=t0, t1=t1, rows=r, prep=prep)


def operands(bits, kind):
    if kind == 2:
        return bits.view(np.float16).astype(np.float64)
    return (bits.astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def sample_rows(res, n=1500, seed=0):
    """Query rows to check: random ones plus the first and last rows of units (256-row blocks), of the row-block halves,
    the rows_full boundary and the last row."""
    q0, q1 = res["q0"], res["q1"]
    nr = q1 - q0 if res["rows"] is None else len(res["rows"])
    rng = np.random.default_rng(seed)
    pick = set(rng.choice(nr, min(n, nr), replace=False).tolist())
    for b in range(0, nr, 128):
        pick.update(x for x in (b, b + 127) if x < nr)
    rf = res["info"]["rows_full"]
    pick.update(x for x in (rf - 1, rf, nr - 1) if 0 <= x < nr)
    return np.array(sorted(pick))


def check_contract(res, n_sample=1500, seed=0):
    """Checks the sampled rows' lists; returns the number of rows checked."""
    inf = res["info"]
    kind = inf["operand_kind"]
    Qop, Top = operands(res["qb"], kind), operands(res["tb"], kind)
    t0, t1 = res["t0"], res["t1"]
    perm = res["perm"].astype(np.int64)
    assert np.array_equal(np.sort(perm), np.arange(len(perm)))
    cols = perm[t0:t1]                     # train-view positions t0..t1-1 -> rows of T
    scale = res["colscale"].astype(np.float64)[cols]
    bias = res["colbias"].astype(np.float64)[cols]
    second = res["rows"] is not None
    cap = 6 if (inf["exact"] and not second) else 8
    picks = sample_rows(res, n_sample, seed)
    qrows = res["rows"][picks] if second else res["q0"] + picks
    Tc = Top[cols]
    Tabs = np.abs(Tc)
    for c0 in range(0, len(picks), 256):  # 256 rows at a time: [rows x columns] float64 blocks
        check_rows(res, picks[c0:c0 + 256], qrows[c0:c0 + 256], Qop, Tc, Tabs, scale, bias, cap, second)
    return len(picks)


def check_rows(res, picks, qrows, Qop, Tc, Tabs, scale, bias, cap, second):
    inf = res["info"]
    t0, t1 = res["t0"], res["t1"]
    ns = inf["nslot"]
    S = (Qop[qrows] @ Tc.T) * scale + bias
    tau = 2e-5 * ((np.abs(Qop[qrows]) @ Tabs.T) * scale + np.abs(bias)) + 1e-30
    for i, (p, q) in enumerate(zip(picks, qrows)):
        read = 1 if (not second and p < inf["rows_full"]) else ns
        ci = res["cidx"][p, :read]
        sc = res["csc"][p, :read]
        assert not (ci == SENT).any() and not np.isnan(sc).any(), (q, ci)          # every slot read was written
        assert (ci[:, cap:] == EMPTY).all() and (sc[:, cap:] == -np.inf).all(), q   # beyond the variant's capacity
        valid = ci[:, :cap] != EMPTY
        assert (sc[:, :cap][~valid] <= -3.0e38).all(), q                              # empty: no real score
        idx = ci[:, :cap][valid].astype(np.int64)
        assert ((idx >= t0) & (idx < t1)).all(), (q, idx)
        assert len(np.unique(idx)) == len(idx), (q, idx)
        key = (sc[:, :cap].view(np.uint32) & np.uint32(0xFFFFFFF8)).view(np.float32).astype(np.float64)
        j = idx - t0
        err = np.abs(key[valid] - S[i, j])
        assert (err <= tau[i, j]).all(), (q, idx[err > tau[i, j]], err.max())
        full = valid.sum(1) == cap
        outside = np.ones(t1 - t0, bool)
        outside[j] = False
        if not full.any():
            assert not outside.any(), (q, "no list is full but columns are missing")
            continue
        W = max(sc[l, :cap].astype(np.float64).min() for l in np.flatnonzero(full))
        bad = np.flatnonzero(outside & (S[i] > W + tau[i]))
        assert bad.size == 0, (q, "columns above W outside every list", bad[:5] + t0, S[i, bad[:5]], W)


def expect(inf, **want):
    got = {k: inf[k] for k in want}
    assert got == want, (inf, want)


def sift_like(rng, n):
    return np.abs(rng.standard_normal((n, 128))).astype(np.float32)


def test_case_a_global_real_valued_balanced_tail(aps):
    G = sm_count(aps)
    X = sift_like(np.random.default_rng(11), 256 * (G + 100))
    res = tc_candidates(aps, None, X, 0)
    print("case a", res["info"])
    expect(res["info"], pre=1, operand_kind=2, exact=0, tail_balanced=2)
    check_contract(res)


def test_case_b_global_integer_merged_tail(aps):
    G = sm_count(aps)
    X = np.random.default_rng(12).integers(0, 256, (256 * (G + 10), 128)).astype(np.float32)
    res = tc_candidates(aps, None, X, 0)
    print("case b", res["info"])
    expect(res["info"], pre=1, operand_kind=2, exact=1, tail_balanced=3)
    check_contract(res)


def flann_real(rng, n):
    """Un-normalised rows, norms spread over 1e-2 .. 1e2."""
    X = rng.standard_normal((n, 128))
    X *= (10.0 ** rng.uniform(-2, 2, n) / np.linalg.norm(X, axis=1))[:, None]
    return X.astype(np.float32)


def test_case_c_flann_real_valued_long_sweep(aps):
    G = sm_count(aps)
    X = flann_real(np.random.default_rng(13), 256 * (G + 10))
    res = tc_candidates(aps, None, X, 1)
    print("case c", res["info"])
    expect(res["info"], pre=1, operand_kind=0, exact=0)
    assert np.any(res["colbias"] != 0)
    check_contract(res)


def test_case_d_flann_integer_long_sweep(aps):
    G = sm_count(aps)
    X = np.random.default_rng(14).integers(0, 256, (256 * (G + 10), 128)).astype(np.float32)
    res = tc_candidates(aps, None, X, 1)
    print("case d", res["info"])
    expect(res["info"], pre=1, operand_kind=0, exact=1)
    check_contract(res)


@pytest.mark.parametrize("prep", [0, 1])
def test_case_e_short_sweep_with_an_empty_segment(aps, prep):
    rng = np.random.default_rng(15 + prep)
    X = sift_like(rng, 600) if prep == 0 else flann_real(rng, 600)
    res = tc_candidates(aps, None, X, prep, q0=0, q1=300)
    inf = res["info"]
    print("case e", prep, inf)
    expect(inf, pre=0, tail_seg=4, units_full=0)
    assert 3 * inf["tiles_per_seg"] >= 5          # the fourth segment starts past the last of the 5 tiles
    assert check_contract(res) == 300


def test_case_f_partial_first_and_last_tiles(aps):
    G = sm_count(aps)
    F = 256 * (G + 10)
    X = sift_like(np.random.default_rng(17), F)
    res = tc_candidates(aps, None, X, 0, q0=77, t0=300, t1=F - 45)
    print("case f", res["info"])
    expect(res["info"], pre=1)
    check_contract(res)


def test_case_g_second_pass_long_sweep(aps):
    F = 50000
    rng = np.random.default_rng(18)
    X = sift_like(rng, F)
    rows = np.sort(rng.choice(F, 3000, replace=False)).astype(np.int32)
    res = tc_candidates(aps, None, X, 0, rows=rows)
    inf = res["info"]
    print("case g", inf)
    expect(inf, pre=1, units_full=0, rows_full=0, nslot=4)
    # rows the launch did not list stay untouched
    assert (res["cidx"][len(rows):] == SENT).all()
    check_contract(res)


def test_case_h_zero_rows_ties_and_constant_rows(aps):
    rng = np.random.default_rng(19)
    X = tcd.degenerate_set(20037, rng)
    res = tc_candidates(aps, None, X, 0)
    print("case h", res["info"])
    expect(res["info"], exact=1)
    zeros = np.flatnonzero((X == 0).all(1))
    assert np.all(res["colscale"][zeros] > 0)
    check_contract(res)


def test_natural_train_order_and_a_query_set(aps):
    """Non-self search (the query side prepared with the train side's flags) on the natural train order."""
    rng = np.random.default_rng(20)
    Q, T = flann_real(rng, 3000), flann_real(rng, 20000)
    res = tc_candidates(aps, Q, T, 1, natural=True)
    assert np.array_equal(res["perm"], np.arange(T.shape[0]))
    check_contract(res)


# ---- end to end: flann_knn_win at long-sweep sizes ----------------------------------------------------------------
def knn(aps, ctx, engine, T, Q, k=4):
    ctx.set_float_engine(engine)
    try:
        idx, dist = aps.flann_knn_win(T, Q, k) if Q is not None else aps.flann_knn_win(T, k)
        st = ctx.last_stats()
    finally:
        ctx.set_float_engine(0)
    return idx, dist, st


@pytest.mark.parametrize("kind,F", [("real", None), ("int", None), ("real", -77)])
def test_flann_long_sweep_self_end_to_end(aps, orc, kind, F):
    G = sm_count(aps)
    n = 256 * (G + 10) + (F or 0)
    rng = np.random.default_rng(21)
    X = flann_real(rng, n) if kind == "real" else rng.integers(0, 256, (n, 128)).astype(np.float32)
    ctx = aps._lib.default_context()
    ti, td, st = knn(aps, ctx, 2, X, None)
    ei, ed, se = knn(aps, ctx, 1, X, None)
    assert st["engine"] == "tcgen05" and se["engine"] == "exact"
    bad = np.flatnonzero((ti != ei).any(1) | (td.view(np.uint32) != ed.view(np.uint32)).any(1))
    assert bad.size == 0, f"{bad.size} rows differ, first {bad[:5]}"
    s = np.sort(rng.choice(n, 1536, replace=False))
    oi, od = orc.knn_l2(X, X[s], 4)
    assert np.array_equal(ti[s], oi) and np.array_equal(td[s].view(np.uint32), od.view(np.uint32))
    print("flann self", kind, n, st, ctx.first_pass_unproven())


def test_flann_query_set_segmented_long_sweep_end_to_end(aps, orc):
    rng = np.random.default_rng(22)
    T, Q = flann_real(rng, 50000), flann_real(rng, 5000)
    ctx = aps._lib.default_context()
    ti, td, st = knn(aps, ctx, 2, T, Q)
    ei, ed, _ = knn(aps, ctx, 1, T, Q)
    assert st["engine"] == "tcgen05"
    assert np.array_equal(ti, ei) and np.array_equal(td.view(np.uint32), ed.view(np.uint32))
    s = np.sort(rng.choice(5000, 1536, replace=False))
    oi, od = orc.knn_l2(T, Q[s], 4)
    assert np.array_equal(ti[s], oi) and np.array_equal(td[s].view(np.uint32), od.view(np.uint32))


# ---- adversarial rounding -----------------------------------------------------------------------------------------
def test_bf16_adversarial_rounding_is_not_proven_with_the_crowd(aps, orc):
    """Each planted query's true neighbours are inflated by ~0.99 of the bf16 term of eps and lie behind a crowd that
    fills every list; a bound below the real error "proves" the crowd.  The rows must go to the second pass or the
    exact search, and the result must be the exact one."""
    X, planted = tcd.flann_adversarial_set()
    maxsq = float((X.astype(np.float64) ** 2).sum(1).max())
    for qt, crowd in planted:
        e_c = tcd.inflation(X[qt[0]], X[crowd], "bf16")
        assert e_c.min() / (tcd.EPS_TERM["bf16"] * maxsq) >= 0.85
    ctx = aps._lib.default_context()
    idx, dist, st = knn(aps, ctx, 2, X, None)
    unproven = ctx.first_pass_unproven()
    oi, od = orc.knn_l2(X, X, 4)
    assert st["engine"] == "tcgen05"
    for qt, _ in planted:
        assert np.array_equal(idx[qt], oi[qt]), (qt, idx[qt], oi[qt])
    assert np.array_equal(idx, oi) and np.array_equal(dist.view(np.uint32), od.view(np.uint32))
    assert unproven + st["fallback_rows"] >= sum(len(qt) for qt, _ in planted)
    print("bf16 adversarial", st, unproven)


def test_fp16_adversarial_rounding_pairwise(aps, orc):
    """The same construction in fp16 through matchFeaturesScratch (|x| <= 2: raw fp16 operands, pair screen in front):
    each planted query's one true neighbour must be found, as the reference finds it.  (These rows do not depend on
    the tensor proof here: the test still passes with the fp16 term of eps halved.)"""
    A, B, planted = tcd.pairwise_adversarial_set()
    maxsq = float(max((A.astype(np.float64) ** 2).sum(1).max(), (B.astype(np.float64) ** 2).sum(1).max()))
    for ra, rb, crowd in planted:
        e_c = tcd.inflation(A[ra], B[crowd], "fp16")
        assert e_c.min() / (tcd.EPS_TERM["fp16"] * maxsq) >= 0.85
    ctx = aps._lib.default_context()
    ctx.set_float_engine(2)
    try:
        m, met = aps.matchFeaturesScratch(A, B, MatchThreshold=3.5, MaxRatio=0.6)
    finally:
        ctx.set_float_engine(0)
    om, omet = orc.match_features(A, B, 3.5, 0.6)
    got = {(int(a) - 1, int(b) - 1) for a, b in m}
    for ra, rb, _ in planted:
        assert (ra, rb) in got, (ra, rb)
    assert np.array_equal(m, om) and np.array_equal(met, omet)
