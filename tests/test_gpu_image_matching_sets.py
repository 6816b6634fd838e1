"""imageMatching over many independent image sets in one call (aps_select_partners_sets + aps_image_matching_sets)
against imageMatching on each set alone with the same seed: candidate pairs, correspondence offsets, model and inverse
bits, inlier masks, n_inliers, accepted and draws_used must be identical.  Also the partner selection per set, the
oracle with given samples, launch counts that do not depend on the number of sets, more than 65535 pairs in one call,
errors, the end-to-end chain from featureMatchingGlobalSets, and the MEX gateway."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
PARAMS = {"maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}
RAW = ("pairs_lin", "pt_ptr", "n_inliers", "accepted", "draws_used", "inliers")


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def _set(aps, n, kp, seed, empty=(), short=0):
    """synthetic ring set; images in `empty` have no keypoints and no matches; `short` cells get 1-3 rows"""
    if n == 0:
        return [], []
    if n == 1:
        return [np.random.default_rng(seed).uniform(0, 2000, (kp, 2))], [[np.zeros((0, 0))]]
    keypoints, matches, _ = aps.synth.synth_matched_keypoints(n, kp, seed=seed)
    for e in empty:
        keypoints[e] = np.zeros((0, 2))
        for k in range(n):
            matches[e][k] = matches[k][e] = np.zeros((0, 0))
    rng = np.random.default_rng(seed + 1)
    for _ in range(short):
        i, j = sorted(rng.choice(n, 2, replace=False))
        if keypoints[i].shape[0] and keypoints[j].shape[0]:
            matches[i][j] = np.asarray(matches[i][j])[:int(rng.integers(1, 4))] if np.size(matches[i][j]) else \
                np.ones((int(rng.integers(1, 4)), 2))
    return keypoints, matches


def _check_sets(aps, inp, ns, kps, ms, seed=3, samples=None, only=None):
    got = aps.imageMatchingSets(inp, ns, kps, ms, seed=seed, samples=samples)
    last = aps.imageMatchingSets.last
    assert len(got) == len(ns)
    for b in (range(len(ns)) if only is None else only):
        gA, gN, gT = got[b]
        if ns[b] < 2:   # no candidate pair: imageMatching returns its empty cells before any RANSAC
            assert last[b]["pairs_lin"].size == 0 and gN.shape == (ns[b], ns[b]) and not gN.any()
            continue
        ref = aps.imageMatching(inp, ns[b], kps[b], ms[b], seed=seed)
        rl = aps.imageMatching.last
        for k in RAW:
            assert np.array_equal(last[b][k], rl[k]), (b, k)
        assert np.array_equal(_bits(last[b]["models"]), _bits(rl["models"])), b
        assert np.array_equal(_bits(last[b]["models_inv"]), _bits(rl["models_inv"])), b
        rA, rN, rT = ref
        assert np.array_equal(gN, rN), b
        n = ns[b]
        for i in range(n):
            for j in range(n):
                assert np.array_equal(np.asarray(gA[i][j]), np.asarray(rA[i][j])), (b, i, j)
                assert (gT[i][j] is None) == (rT[i][j] is None), (b, i, j)
                if gT[i][j] is not None:
                    assert np.array_equal(_bits(gT[i][j]), _bits(rT[i][j])), (b, i, j)
    return got, last


def test_small_sets_equal_the_single_set_call(aps):
    """64 sets of 6 images and 300 sets of 3 images, mixed with empty, one-image and zero-keypoint sets and pairs with
    fewer than 4 correspondences"""
    for B, n, kp in ((64, 6, 300), (300, 3, 200)):
        ns, kps, ms = [], [], []
        for b in range(B):
            nb = {5: 0, 17: 1, 40: 2}.get(b, n)
            k, m = _set(aps, nb, kp, 1000 * n + b, empty=(0,) if b == 23 else (), short=2 if b % 7 == 0 else 0)
            ns.append(nb), kps.append(k), ms.append(m)
        _, last = _check_sets(aps, PARAMS, ns, kps, ms)
        assert sum(last[b]["accepted"].sum() for b in range(B) if "accepted" in last[b]) >= B


def test_c1_shaped_sets_equal_the_single_set_call(aps):
    """C1 shape: 6 images of 2048 keypoints, one image empty; 8 such sets with different seeds and maxIter"""
    ns, kps, ms = [], [], []
    for b in range(8):
        k, m = _set(aps, 6, 2048, 500 + b, empty=(3,))
        ns.append(6), kps.append(k), ms.append(m)
    _check_sets(aps, PARAMS, ns, kps, ms, seed=11)
    _check_sets(aps, dict(PARAMS, maxIter=100, maxDistance=2.0, mBrownLowe=2), ns, kps, ms, seed=12)


def test_partner_selection_equals_single_set_call(aps):
    rng = np.random.default_rng(4)
    sets = []
    for b in range(120):
        n = int(rng.integers(0, 12))
        sets.append(rng.integers(0, 3, (n, n)) * int(rng.integers(1, 4)))   # tie-heavy: few distinct values
    for m in (1, 2, 4, 6, 11, 40):
        got = aps.selectImagePartnersSets(sets, m)
        for c, (cand, lin) in zip(sets, got):
            if c.shape[0] == 0:
                assert cand.shape == (0, 0) and lin.size == 0
                continue
            rc, rl = aps.selectImagePartners(c, m)
            assert np.array_equal(cand, rc) and np.array_equal(lin, rl)


def test_given_samples_equal_device_draws_and_the_oracle(aps, orc):
    """per-set aps_ransac_sample_table tables: the same result as drawing on the device (keys per set), and the
    oracle's RANSAC on a few sets"""
    ns, kps, ms = [], [], []
    for b in range(6):
        k, m = _set(aps, 5, 400, 77 + b)
        ns.append(5), kps.append(k), ms.append(m)
    drawn = aps.imageMatchingSets(PARAMS, ns, kps, ms, seed=9)
    last = [dict(d) for d in aps.imageMatchingSets.last]
    tabs = [aps.ransacSampleTable(last[b]["pt_ptr"], 1000, seed=9) for b in range(len(ns))]
    given = aps.imageMatchingSets(PARAMS, ns, kps, ms, seed=123, samples=tabs)
    for b in range(len(ns)):
        g = aps.imageMatchingSets.last[b]
        for k in RAW:
            assert np.array_equal(g[k], last[b][k]), (b, k)
        assert np.array_equal(_bits(g["models"]), _bits(last[b]["models"]))
        assert np.array_equal(drawn[b][1], given[b][1])
    for b in (0, 3, 5):
        n, lin, ptr = ns[b], last[b]["pairs_lin"], last[b]["pt_ptr"]
        P1 = np.vstack([kps[b][c // n][np.asarray(ms[b][c % n][c // n], np.int64)[:, 1] - 1] for c in lin])
        P2 = np.vstack([kps[b][c % n][np.asarray(ms[b][c % n][c // n], np.int64)[:, 0] - 1] for c in lin])
        o = orc.image_matching_batch(ptr, P1, P2, 5.5, 99.9, 500, tabs[b])
        g = aps.imageMatchingSets.last[b]
        assert np.array_equal(o["inliers"], g["inliers"]) and np.array_equal(o["accepted"], g["accepted"])
        assert np.array_equal(o["n_inliers"], g["n_inliers"]) and np.array_equal(o["draws_used"], g["draws_used"])
        acc = o["accepted"]
        assert acc.sum() >= 2
        assert np.allclose(g["models"][acc], o["models"][acc], rtol=1e-9, atol=1e-12)


def test_launch_count_does_not_depend_on_the_number_of_sets(aps):
    L = aps._lib.lib()
    counts = []
    for B in (2, 200):
        ns, kps, ms = [], [], []
        for b in range(B):
            k, m = _set(aps, 4, 150, 9000 + b)
            ns.append(4), kps.append(k), ms.append(m)
        aps.imageMatchingSets(PARAMS, ns, kps, ms)
        c0 = L.aps_launch_count()
        aps.imageMatchingSets(PARAMS, ns, kps, ms)
        counts.append(L.aps_launch_count() - c0)
    assert counts[0] == counts[1] and counts[0] <= 3 + 12, counts


def test_more_than_65535_pairs_in_one_call(aps):
    """22000 sets of 3 images (3 candidate pairs each, 66000 in all) with a few correspondences per pair: the chain runs
    in two chunks; sets on both sides of the chunk boundary equal their single-set calls"""
    rng = np.random.default_rng(8)
    B, n, kp = 22000, 3, 8
    ns, kps, ms = [n] * B, [], []
    for b in range(B):
        kps.append([rng.uniform(0, 500, (kp, 2)) for _ in range(n)])
        m = [[np.zeros((0, 0))] * n for _ in range(n)]
        for i in range(n):
            for j in range(i + 1, n):
                m[i][j] = rng.integers(1, kp + 1, (int(rng.integers(2, 9)), 2)).astype(np.float64)
        ms.append(m)
    inp = dict(PARAMS, maxIter=4)
    got, last = _check_sets(aps, inp, ns, kps, ms, seed=5, only=[0, 1, 9999, 21844, 21845, 21846, B - 1])
    assert sum(last[b]["pairs_lin"].size for b in range(B)) == 3 * B


def test_match_index_out_of_range_in_one_set_fails_the_call(aps):
    ns, kps, ms = [], [], []
    for b in range(3):
        k, m = _set(aps, 4, 100, 40 + b)
        ns.append(4), kps.append(k), ms.append(m)
    bad = np.array(ms[1][0][1], copy=True)
    bad[2, 1] = 101
    ms[1][0][1] = bad
    with pytest.raises(aps.ApsError) as e:
        aps.imageMatchingSets(PARAMS, ns, kps, ms)
    assert e.value.identifier == "refineMatch:MatchIndexOutOfBounds" and "set 2" in e.value.message


def test_feature_matching_global_sets_then_image_matching_sets(aps):
    """featureMatchingGlobalSets -> imageMatchingSets equals featureMatchingGlobal -> imageMatching set by set"""
    desc, c = aps.synth.make_config(1, n=6, kp=700)
    sets = [desc[:4], desc[4:6], desc[1:5], desc[2:3]]
    rng = np.random.default_rng(2)
    kps = [[rng.uniform(0, 2000, (d.shape[0], 2)) for d in s] for s in sets]
    ns = [len(s) for s in sets]
    inp = dict(PARAMS, k=c["k"], Ratiothreshold=c["ratio"], mBrownLowe=2, maxDistance=1e6)
    matches = aps.featureMatchingGlobalSets(inp, sets, ns)
    got = aps.imageMatchingSets(inp, ns, kps, matches, seed=6)
    for b in range(len(sets)):
        mb = aps.featureMatchingGlobal(inp, sets[b], ns[b])
        rA, rN, rT = aps.imageMatching(inp, ns[b], kps[b], mb, seed=6)
        gA, gN, gT = got[b]
        assert np.array_equal(gN, rN)
        for i in range(ns[b]):
            for j in range(ns[b]):
                assert np.array_equal(np.asarray(gA[i][j]), np.asarray(rA[i][j]))
                assert (gT[i][j] is None) == (rT[i][j] is None)
    assert any(g[1].any() for g in got)


def test_gateway_real_call_equals_host_mirror(tmp_path):
    import test_mex_gateways as tg

    pkg = __import__("__graft_entry__").load_package()
    ns, kps, ms = [], [], []
    for b, n in enumerate((4, 1, 3, 5)):
        k, m = _set(pkg, n, 250, 60 + b)
        ns.append(n), kps.append(k), ms.append(m)
    mats = []
    for n, k, m in zip(ns, kps, ms):
        mats += [(2, np.asarray(x, np.float64).reshape(-1, 2)) for x in k]
        mats += [(2, np.asarray(m[c % n][c // n], np.float64).reshape(-1, 2) if np.size(m[c % n][c // n])
                  else np.zeros((0, 0))) for c in range(n * n)]
    inp = dict(PARAMS, mBrownLowe=3)
    outs = tg._run_gate("gate_imatch_sets", mats, [len(ns)] + ns + [3, 5.5, 99.9, 500, 0], tmp_path)
    ref = pkg.imageMatchingSets(inp, ns, kps, ms, seed=0)
    o = 0
    for b, n in enumerate(ns):
        rA, rN, rT = ref[b]
        for c in range(n * n):
            want, got = np.asarray(rA[c % n][c // n]), outs[o + c]
            assert (got is None and want.size == 0) or np.array_equal(got, want), (b, c)
        o += n * n
        assert np.array_equal(outs[o], rN), b
        o += 1
        for c in range(n * n):
            want, got = rT[c % n][c // n], outs[o + c]
            assert (got is None) == (want is None) and (want is None or np.array_equal(got, want)), (b, c)
        o += n * n
    assert any(r[1].any() for r in ref)
