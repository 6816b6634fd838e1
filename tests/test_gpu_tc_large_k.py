"""GPU: the tensor kNN path for 6 <= k <= 12 (K' = 16 candidates per list, up to 64 per row in the re-rank).

End to end, every result must equal the oracle or the exact CUDA-core engine bit for bit.  The candidate lists of the
K' = 16 kernel variants are checked against the contract of the re-rank's completeness proof (aps_rerank.cu): every
slot the re-rank reads was written, every train column in none of the row's lists scores at most W (the largest
minimum retained score over the row's full lists), and a list that is not full holds every column of its range."""
import numpy as np
import pytest

import tc_contract_data as tcd

pytestmark = pytest.mark.gpu

SENT = 0xA5A5A5A5
EMPTY = 0xFFFFFFFF
KC = 16
INFO = ("sm_count", "nslot", "rows_full", "exact", "operand_kind", "pre", "units_full", "tail_units", "tail_seg",
        "tail_balanced", "tiles_per_seg", "kcand")


def sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


def knn(aps, ctx, engine, T, Q, k):
    ctx.set_float_engine(engine)
    try:
        idx, dist = aps.flann_knn_win(T, Q, k) if Q is not None else aps.flann_knn_win(T, k)
        st = ctx.last_stats()
        unproven = ctx.first_pass_unproven()
    finally:
        ctx.set_float_engine(0)
    return idx, dist, st, unproven


def same_bits(a, b):
    return np.array_equal(a[0], b[0]) and np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32))


# ---- flann_knn_win ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [6, 8, 12, 13])
def test_flann_knn_float_large_k_vs_oracle(aps, orc, k):
    """k <= 12 runs on the tensor path (auto engine), k = 13 on the exact engine."""
    rng = np.random.default_rng(100 + k)
    X = rng.standard_normal((5000, 128)).astype(np.float32)
    X[10:14] = X[10]
    ctx = aps._lib.default_context()
    idx, dist, st, _ = knn(aps, ctx, 0, X, X[:900].copy(), k)
    assert st["engine"] == ("tcgen05" if k <= 12 else "exact"), st
    oi, od = orc.knn_l2(X, X[:900], k)
    assert same_bits((idx, dist), (oi, od))


def test_flann_knn_query_set_k10_bf16(aps, orc):
    rng = np.random.default_rng(110)
    T = rng.standard_normal((6000, 128)).astype(np.float32)
    Q = (rng.standard_normal((1200, 128)) * 1.3).astype(np.float32)
    ctx = aps._lib.default_context()
    idx, dist, st, _ = knn(aps, ctx, 0, T, Q, 10)
    assert st["engine"] == "tcgen05"
    oi, od = orc.knn_l2(T, Q, 10)
    assert same_bits((idx, dist), (oi, od))


# ---- featureMatchingGlobal / GlobalPlan ---------------------------------------------------------------------------
@pytest.mark.parametrize("k", [8, 12])
def test_global_float_c1_large_k(aps, orc, k):
    desc, c = aps.synth.make_config(1)
    ref = orc.feature_matching_global(desc, k, c["ratio"])
    got = aps.featureMatchingGlobal({"k": k, "Ratiothreshold": c["ratio"]}, desc, len(desc))
    assert aps._lib.default_context().last_stats()["engine"] == "tcgen05"
    rows = 0
    for j in range(len(desc)):
        for i in range(j):
            exp = ref["cells"].get((i, j))
            if exp is None:
                assert got[i][j].size == 0, (i, j)
            else:
                assert got[i][j].shape == exp.shape and (got[i][j] == exp).all(), (i, j)
                rows += len(exp)
    assert rows == len(ref["rows"]) and rows > 0


def plan_table(aps, ctx, desc, engine, k, q_ranges=None):
    ctx.set_float_engine(engine)
    try:
        plan = aps.GlobalPlan(ctx, [d.shape[0] for d in desc], desc[0].shape[1], False, k)
        plan.upload(desc)
        plan.prepare()
        ranges = q_ranges or [(0, plan.F)]
        unproven = []
        for q0, q1 in ranges:
            plan.knn(q0, q1)
            unproven.append(ctx.first_pass_unproven())
        idx, dist = plan.download_knn()
        stats = ctx.last_stats()
        plan.close()
    finally:
        ctx.set_float_engine(0)
    return (idx, dist), stats, unproven


@pytest.mark.parametrize("cid", [2, 6])
def test_full_size_k12_tensor_equals_exact(aps, cid):
    """Every row of C2 (integer SIFT) and of its real-valued twin (config 6) at k = 12.  On config 6 the first proof
    leaves more rows open than the exact engine takes directly, so the 64-candidate second pass runs."""
    ctx = aps._lib.default_context()
    desc, _ = aps.synth.make_config(cid)
    tc, st_tc, (unproven,) = plan_table(aps, ctx, desc, 0, 12)
    ex, st_ex, _ = plan_table(aps, ctx, desc, 1, 12)
    print(f"config {cid} k=12: first_pass_unproven={unproven} fallback_rows={st_tc['fallback_rows']}")
    assert st_tc["engine"] == "tcgen05" and st_ex["engine"] == "exact"
    bad = np.flatnonzero((tc[0] != ex[0]).any(1) | (tc[1].view(np.uint32) != ex[1].view(np.uint32)).any(1))
    assert bad.size == 0, f"{bad.size} of {tc[0].shape[0]} rows differ, first {bad[:5]}"
    if cid == 6:
        assert unproven > 128  # k_route_unproven's short-list limit: above it the second tensor pass runs


def test_global_plan_k8_two_query_shards(aps):
    ctx = aps._lib.default_context()
    desc, _ = aps.synth.make_config(1)
    F = sum(d.shape[0] for d in desc)
    q = 5000
    one, st, _ = plan_table(aps, ctx, desc, 0, 8)
    two, _, _ = plan_table(aps, ctx, desc, 0, 8, [(0, q), (q, F)])
    assert st["engine"] == "tcgen05"
    assert same_bits(one, two)


# ---- adversarial inputs -------------------------------------------------------------------------------------------
def test_bf16_adversarial_set_k8_equals_exact(aps):
    X, _ = tcd.flann_adversarial_set()
    ctx = aps._lib.default_context()
    ti, td, st, unproven = knn(aps, ctx, 2, X, None, 8)
    ei, ed, se, _ = knn(aps, ctx, 1, X, None, 8)
    assert st["engine"] == "tcgen05" and se["engine"] == "exact"
    assert same_bits((ti, td), (ei, ed))
    print("bf16 adversarial k=8", st, unproven)


def test_identical_crowd_k12_falls_back(aps, orc):
    """72 identical rows, more than the 4 lists of 16 a row can have: whatever the schedule, some list of every crowd
    row holds crowd members only, so its worst retained distance is within eps of 0 = the row's 12th exact distance,
    and the row cannot be proven by the first pass.  The lists are checked for that, the first pass must leave at
    least the 72 crowd rows open, and the result must be the oracle's."""
    rng = np.random.default_rng(120)
    X = rng.standard_normal((5000, 128)).astype(np.float32)
    crowd = rng.choice(5000, 72, replace=False)
    X[crowd] = X[crowd[0]]
    res = tc_candidates(aps, None, X, 1, k=12)  # flann_knn_win's preparation and schedule for this search
    assert res["info"]["kcand"] == KC and res["info"]["nslot"] <= 4
    in_crowd = np.zeros(len(X), bool)
    in_crowd[crowd] = True
    for p in crowd:
        read = 1 if p < res["info"]["rows_full"] else res["info"]["nslot"]
        lists = res["cidx"][p, :read]
        crowd_only = [(l != EMPTY).all() and in_crowd[res["perm"][l.astype(np.int64)]].all() for l in lists]
        assert any(crowd_only), (p, lists)
    ctx = aps._lib.default_context()
    idx, dist, st, unproven = knn(aps, ctx, 2, X, None, 12)
    assert st["engine"] == "tcgen05"
    assert unproven >= len(crowd), (unproven, st)
    oi, od = orc.knn_l2(X, X, 12)
    assert same_bits((idx, dist), (oi, od))
    print("identical crowd k=12", st, unproven)


# ---- the candidate lists against the re-rank's contract -----------------------------------------------------------
def tc_candidates(aps, Q, T, prep, q0=0, q1=None, t0=0, t1=None, rows=None, natural=False, k=8):
    ctx = aps._lib.default_context()
    L = aps._lib.lib()
    T = np.ascontiguousarray(T, np.float32)
    Q = T if Q is None else np.ascontiguousarray(Q, np.float32)
    nq, nt, D = Q.shape[0], T.shape[0], T.shape[1]
    q1 = nq if q1 is None else q1
    t1 = nt if t1 is None else t1
    nr = q1 - q0
    cidx = np.zeros(nr * 64, np.uint32)
    csc = np.zeros(nr * 64, np.float32)
    perm = np.zeros(nt, np.int32)
    qb = np.zeros((nq, D), np.uint16)
    tb = np.zeros((nt, D), np.uint16)
    cs = np.zeros(nt, np.float32)
    cb = np.zeros(nt, np.float32)
    info = np.zeros(12, np.int64)
    r = None if rows is None else np.ascontiguousarray(rows, np.int32)
    aps._lib.check(L.aps_debug_tc_candidates_k(
        ctx.handle, Q.ctypes.data, nq, T.ctypes.data, nt, D, prep, int(natural), q0, q1, t0, t1,
        None if r is None else r.ctypes.data, 0 if r is None else len(r), cidx.ctypes.data, csc.ctypes.data,
        perm.ctypes.data, qb.ctypes.data, tb.ctypes.data, cs.ctypes.data, cb.ctypes.data, info.ctypes.data, k))
    inf = dict(zip(INFO, info.tolist()))
    ns, kc = inf["nslot"], inf["kcand"]
    return dict(info=inf, cidx=cidx[:nr * ns * kc].reshape(nr, ns, kc), csc=csc[:nr * ns * kc].reshape(nr, ns, kc),
                sent_tail=cidx[nr * ns * kc:], perm=perm, qb=qb, tb=tb, colscale=cs, colbias=cb, q0=q0, q1=q1, t0=t0,
                t1=t1, rows=r)


def operands(bits, kind):
    if kind == 2:
        return bits.view(np.float16).astype(np.float64)
    return (bits.astype(np.uint32) << 16).view(np.float32).astype(np.float64)


def sample_rows(res, n=1200, seed=0):
    nr = res["q1"] - res["q0"] if res["rows"] is None else len(res["rows"])
    rng = np.random.default_rng(seed)
    pick = set(rng.choice(nr, min(n, nr), replace=False).tolist())
    for b in range(0, nr, 128):
        pick.update(x for x in (b, b + 127) if x < nr)
    rf = res["info"]["rows_full"]
    pick.update(x for x in (rf - 1, rf, nr - 1) if 0 <= x < nr)
    return np.array(sorted(pick))


def segment_ranges(res):
    """Column range of each list of a fully segmented schedule (short sweeps, second pass): list s covers the train tiles
    [tile_lo + s * tiles_per_seg, ...) cut to [t0, t1); None when the schedule is not of that form."""
    inf = res["info"]
    if inf["units_full"] != 0 or inf["tail_balanced"] != 0:
        return None
    t0, t1, tps = res["t0"], res["t1"], inf["tiles_per_seg"]
    lo = t0 // 128
    return [(max(t0, (lo + s * tps) * 128), min(t1, (lo + (s + 1) * tps) * 128)) for s in range(inf["nslot"])]


def check_contract(res, n_sample=1200, seed=0):
    """Checks the sampled rows' lists; returns the number of rows checked."""
    inf = res["info"]
    assert inf["kcand"] == KC, inf
    kind = inf["operand_kind"]
    Qop, Top = operands(res["qb"], kind), operands(res["tb"], kind)
    t0, t1 = res["t0"], res["t1"]
    perm = res["perm"].astype(np.int64)
    assert np.array_equal(np.sort(perm), np.arange(len(perm)))
    cols = perm[t0:t1]
    scale = res["colscale"].astype(np.float64)[cols]
    bias = res["colbias"].astype(np.float64)[cols]
    second = res["rows"] is not None
    picks = sample_rows(res, n_sample, seed)
    qrows = res["rows"][picks] if second else res["q0"] + picks
    Tc = Top[cols]
    Tabs = np.abs(Tc)
    seg = segment_ranges(res)
    for c0 in range(0, len(picks), 256):
        p, q = picks[c0:c0 + 256], qrows[c0:c0 + 256]
        S = (Qop[q] @ Tc.T) * scale + bias
        tau = 2e-5 * ((np.abs(Qop[q]) @ Tabs.T) * scale + np.abs(bias)) + 1e-30
        for i in range(len(p)):
            check_row(res, p[i], q[i], S[i], tau[i], second, seg)
    return len(picks)


def check_row(res, p, q, S, tau, second, seg):
    inf = res["info"]
    t0, t1 = res["t0"], res["t1"]
    read = 1 if (not second and p < inf["rows_full"]) else inf["nslot"]
    ci = res["cidx"][p, :read]
    sc = res["csc"][p, :read]
    assert not (ci == SENT).any() and not np.isnan(sc).any(), (q, ci)       # every slot read was written
    valid = ci != EMPTY
    assert (sc[~valid] <= -3.0e38).all(), q                                    # empty: no real score
    idx = ci[valid].astype(np.int64)
    assert ((idx >= t0) & (idx < t1)).all(), (q, idx)
    assert len(np.unique(idx)) == len(idx), (q, idx)
    key = (sc.view(np.uint32) & np.uint32(0xFFFFFFF0)).view(np.float32).astype(np.float64)  # 4 slot bits
    err = np.abs(key[valid] - S[idx - t0])
    assert (err <= tau[idx - t0]).all(), (q, err.max())
    full = valid.sum(1) == KC
    outside = np.ones(t1 - t0, bool)
    outside[idx - t0] = False
    for l in np.flatnonzero(~full):                                            # a list that is not full holds its range
        if read == 1:
            lo, hi = t0, t1
        elif seg is not None:
            lo, hi = seg[l]
        else:
            continue
        held = np.zeros(t1 - t0, bool)
        held[ci[l][valid[l]].astype(np.int64) - t0] = True
        assert held[lo - t0:hi - t0].all() if hi > lo else True, (q, l, lo, hi)
    if not full.any():
        assert not outside.any(), (q, "no list is full but columns are missing")
        return
    W = max(sc[l].astype(np.float64).min() for l in np.flatnonzero(full))
    bad = np.flatnonzero(outside & (S > W + tau))
    assert bad.size == 0, (q, "columns above W outside every list", bad[:5] + t0, S[bad[:5]], W)


def expect(inf, **want):
    got = {k: inf[k] for k in want}
    assert got == want, (inf, want)


def sift_like(rng, n):
    return np.abs(rng.standard_normal((n, 128))).astype(np.float32)


def flann_real(rng, n):
    X = rng.standard_normal((n, 128))
    X *= (10.0 ** rng.uniform(-2, 2, n) / np.linalg.norm(X, axis=1))[:, None]
    return X.astype(np.float32)


@pytest.mark.parametrize("case", ["fp16_real_balanced", "fp16_integer_merged", "bf16_real_long", "bf16_integer_long"])
def test_contract_long_sweeps(aps, case):
    G = sm_count()
    rng = np.random.default_rng(200 + len(case))
    if case == "fp16_real_balanced":
        X, prep, want = sift_like(rng, 256 * (G + 100)), 0, dict(pre=1, operand_kind=2, tail_balanced=2)
    elif case == "fp16_integer_merged":
        X = rng.integers(0, 256, (256 * (G + 10), 128)).astype(np.float32)
        prep, want = 0, dict(pre=1, operand_kind=2, exact=1, tail_balanced=3)
    elif case == "bf16_real_long":
        X, prep, want = flann_real(rng, 256 * (G + 10)), 1, dict(pre=1, operand_kind=0, exact=0)
    else:
        X = rng.integers(0, 256, (256 * (G + 10), 128)).astype(np.float32)
        prep, want = 1, dict(pre=1, operand_kind=0, exact=1)
    res = tc_candidates(aps, None, X, prep)
    print(case, res["info"])
    expect(res["info"], kcand=KC, **want)
    check_contract(res)


@pytest.mark.parametrize("prep", [0, 1])
def test_contract_short_sweep_with_an_empty_segment(aps, prep):
    rng = np.random.default_rng(215 + prep)
    X = sift_like(rng, 600) if prep == 0 else flann_real(rng, 600)
    res = tc_candidates(aps, None, X, prep, q0=0, q1=300)
    inf = res["info"]
    print("short sweep", prep, inf)
    expect(inf, pre=0, tail_seg=4, units_full=0, kcand=KC)
    assert 3 * inf["tiles_per_seg"] >= 5          # the fourth segment starts past the last of the 5 tiles
    assert check_contract(res) == 300


def test_contract_partial_first_and_last_tiles(aps):
    G = sm_count()
    F = 256 * (G + 10)
    X = sift_like(np.random.default_rng(217), F)
    res = tc_candidates(aps, None, X, 0, q0=77, t0=300, t1=F - 45)
    print("partial tiles", res["info"])
    expect(res["info"], pre=1, kcand=KC)
    check_contract(res)


@pytest.mark.parametrize("prep", [0, 1])
def test_contract_second_pass(aps, prep):
    F = 50000
    rng = np.random.default_rng(218 + prep)
    X = sift_like(rng, F) if prep == 0 else flann_real(rng, F)
    rows = np.sort(rng.choice(F, 3000, replace=False)).astype(np.int32)
    res = tc_candidates(aps, None, X, prep, rows=rows)
    inf = res["info"]
    print("second pass", prep, inf)
    expect(inf, pre=1, units_full=0, rows_full=0, nslot=4, kcand=KC)
    assert (res["cidx"][len(rows):] == SENT).all() and (res["sent_tail"] == SENT).all()  # unlisted rows untouched
    check_contract(res)


def test_k4_lists_keep_eight_candidates(aps):
    """k <= 5 keeps K' = 8 through the same entry (the old entry point is this one with k = 4)."""
    X = sift_like(np.random.default_rng(219), 600)
    res = tc_candidates(aps, None, X, 0, q0=0, q1=300, k=5)
    assert res["info"]["kcand"] == 8
