"""featureMatchingGlobal + imageMatching in one call (aps_global_image_matching[_sets]) against the two-call chains at
the same seed: featureMatchingGlobalSets -> imageMatchingSets, and featureMatchingGlobal -> imageMatching set by set.
Candidate pairs, correspondence offsets, n_inliers, accepted, draws_used, the bits of the models and their inverses,
allMatches, numMatches and tforms must be identical, and return_matches must give featureMatchingGlobalSets' lists.
Also launch counts that do not depend on the number of sets, more than 65535 candidate pairs, and the MEX gateway."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
PARAMS = {"k": 4, "Ratiothreshold": 0.8, "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500,
          "mBrownLowe": 6}
KEYS = ("pairs_lin", "pt_ptr", "n_inliers", "accepted", "draws_used")


def _bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def make_set(aps, rng, n, kp, kind="sift", empty=(), share=0.3, consistent=0.75):
    """n images on a ring.  Image i receives noisy copies of share * kp descriptor rows of the previous live image, and
    the keypoints of those rows are a random mild homography of the source rows' keypoints (+ 0.5 px noise) for a pair
    drawn consistent, or left random otherwise: consistent pairs pass RANSAC, the others and the stray pairs do not.
    Returns (descriptor cells, keypoints)."""
    D = 32 if kind == "orb" else 128
    live = [i for i in range(n) if i not in empty]
    s = int(share * kp)
    if kind == "orb":
        desc = {i: rng.integers(0, 256, (kp, D), dtype=np.uint8) for i in live}
    else:
        desc = {i: np.abs(rng.standard_normal((kp, D))) / 11.0 for i in live}
    kps = {i: rng.uniform(0.0, 2000.0, (kp, 2)) for i in live}
    for pos, i in enumerate(live):
        src = live[pos - 1]
        if len(live) < 2 or src == i or s == 0:
            continue
        rows = s + rng.permutation(kp - s)[:s]   # sources come from rows no image writes into
        if kind == "orb":
            desc[i][:s] = desc[src][rows] ^ np.packbits(rng.random((s, 8 * D)) < 0.03, axis=1)
        else:
            desc[i][:s] = desc[src][rows] + rng.normal(0.0, 0.002, (s, D))
        if rng.random() < consistent:
            H = np.eye(3) + rng.normal(0.0, 1.0, (3, 3)) * np.array([[0.05, 0.05, 60.0], [0.05, 0.05, 60.0],
                                                                      [2e-5, 2e-5, 0.0]])
            q = np.c_[kps[src][rows], np.ones(s)] @ H.T
            kps[i][:s] = q[:, :2] / q[:, 2:3] + rng.normal(0.0, 0.5, (s, 2))
    cells, kpl = [], []
    for i in range(n):
        if i not in desc:
            cells.append(aps.binaryFeatures(np.zeros((0, D), np.uint8)) if kind == "orb" else np.zeros((0, D), np.float32))
            kpl.append(np.zeros((0, 2)))
            continue
        d = desc[i]
        cells.append(aps.binaryFeatures(d) if kind == "orb" else aps.synth._sift_quantise(d))
        kpl.append(kps[i])
    return cells, kpl


def _same_cells(a, b, n):
    for i in range(n):
        for j in range(n):
            assert np.array_equal(np.asarray(a[i][j]), np.asarray(b[i][j])), (i, j)


def _same_result(got, glast, ref, rlast, n):
    for k in KEYS:
        if k in rlast:
            assert np.array_equal(glast[k], rlast[k]), k
    if "models" in rlast:
        assert np.array_equal(_bits(glast["models"]), _bits(rlast["models"]))
        assert np.array_equal(_bits(glast["models_inv"]), _bits(rlast["models_inv"]))
    (gA, gN, gT), (rA, rN, rT) = got, ref
    assert np.array_equal(gN, rN)
    _same_cells(gA, rA, n)
    for i in range(n):
        for j in range(n):
            assert (gT[i][j] is None) == (rT[i][j] is None), (i, j)
            if gT[i][j] is not None:
                assert np.array_equal(_bits(gT[i][j]), _bits(rT[i][j])), (i, j)


def check_against_chains(aps, inp, cells, kps, seed=3, single=None):
    """the fused call against both chains; single: sets also compared with the one-set chain (default all).
    Returns (accepted pairs, candidate pairs)."""
    ns = [len(c) for c in cells]
    got, lists = aps.globalImageMatchingSets(inp, cells, ns, kps, seed=seed, return_matches=True)
    glast = aps.globalImageMatchingSets.last
    matches = aps.featureMatchingGlobalSets(inp, cells, ns)
    ref = aps.imageMatchingSets(inp, ns, kps, matches, seed=seed)
    rlast = aps.imageMatchingSets.last
    for b, n in enumerate(ns):
        _same_cells(lists[b], matches[b], n)
        _same_result(got[b], glast[b], ref[b], rlast[b], n)
    for b in (range(len(ns)) if single is None else single):
        mb = aps.featureMatchingGlobal(inp, cells[b], ns[b])
        r1 = aps.imageMatching(inp, ns[b], kps[b], mb, seed=seed)
        _same_result(got[b], glast[b], r1, aps.imageMatching.last if glast[b]["pairs_lin"].size else {}, ns[b])
        g1, m1 = aps.globalImageMatching(inp, cells[b], ns[b], kps[b], seed=seed, return_matches=True)
        _same_result(g1, aps.globalImageMatching.last, r1, glast[b], ns[b])
        _same_cells(m1, mb, ns[b])
    acc = sum(int(l["accepted"].sum()) for l in glast)
    return acc, sum(l["pairs_lin"].size for l in glast)


@pytest.mark.parametrize("extra", [{}, {"apsMutual": 1}, {"k": 8}])
def test_mixed_batch_equals_both_chains(aps, extra):
    """exact-path sets first, tensor-path sets (>= 2048 rows) after them, so the pass order differs from the set order;
    with a set without descriptors, a one-image set and images without descriptors"""
    rng = np.random.default_rng(11)
    shapes = [(4, 300, ()), (3, 900, ()), (2, 200, (0, 1)), (1, 400, ()), (5, 250, (2,)), (4, 700, (1,)), (3, 150, ())]
    cells, kps = [], []
    for n, kp, empty in shapes:
        c, k = make_set(aps, rng, n, kp, empty=empty)
        cells.append(c), kps.append(k)
    acc, cand = check_against_chains(aps, dict(PARAMS, **extra), cells, kps)
    assert 0 < acc < cand, (acc, cand)


def test_orb_sets_equal_both_chains(aps):
    rng = np.random.default_rng(12)
    cells, kps = [], []
    for n, kp, empty in ((4, 400, ()), (3, 300, (2,)), (1, 100, ()), (5, 500, ())):
        c, k = make_set(aps, rng, n, kp, kind="orb", empty=empty)
        cells.append(c), kps.append(k)
    acc, cand = check_against_chains(aps, dict(PARAMS, BFMatch=1), cells, kps)
    assert 0 < acc < cand, (acc, cand)


@pytest.mark.parametrize("shape", [(6, 2048, (3,)), (20, 8192, ())], ids=["C1", "C2"])
def test_single_c1_and_c2_shaped_sets(aps, shape):
    n, kp, empty = shape
    cells, kps = make_set(aps, np.random.default_rng(13), n, kp, empty=empty)
    acc, cand = check_against_chains(aps, PARAMS, [cells], [kps], seed=7)
    assert 0 < acc < cand, (acc, cand)


def test_launch_count_does_not_depend_on_the_number_of_sets(aps):
    L = aps._lib.lib()
    counts = []
    for B in (2, 200):
        rng = np.random.default_rng(14)
        cells, kps = zip(*[make_set(aps, rng, 4, 120) for _ in range(B)])
        aps.globalImageMatchingSets(PARAMS, list(cells), [4] * B, list(kps))
        c0 = L.aps_launch_count()
        aps.globalImageMatchingSets(PARAMS, list(cells), [4] * B, list(kps))
        counts.append(L.aps_launch_count() - c0)
    assert counts[0] == counts[1], counts


def test_more_than_65535_candidate_pairs(aps):
    """22000 sets of 3 images sharing rows (3 candidate pairs each, 66000 in all): the RANSAC runs in two chunks"""
    rng = np.random.default_rng(15)
    B = 22000
    cells, kps = zip(*[make_set(aps, rng, 3, 16, share=0.5) for _ in range(B)])
    inp = dict(PARAMS, maxIter=4)
    acc, cand = check_against_chains(aps, inp, list(cells), list(kps), seed=5, single=[0, 1, 21844, 21845, B - 1])
    assert cand > 65535 and 0 < acc < cand, (acc, cand)


def test_gateway_real_call_equals_host_mirror(tmp_path):
    import test_mex_gateways as tg

    pkg = __import__("__graft_entry__").load_package()
    rng = np.random.default_rng(16)
    sets = [make_set(pkg, rng, n, kp, empty=e) for n, kp, e in ((4, 300, ()), (1, 100, ()), (3, 700, (1,)))]
    ns = [len(c) for c, _ in sets]
    mats = []
    for c, k in sets:
        mats += [(0, np.asarray(d, np.float32).reshape(-1, 128)) for d in c]
        mats += [(2, np.asarray(x, np.float64).reshape(-1, 2)) for x in k]
    inp = dict(PARAMS, mBrownLowe=3)
    outs = tg._run_gate("gate_gimatch", mats, [len(ns)] + ns + [4, 0.8, 3, 5.5, 99.9, 500, 0], tmp_path)
    ref = pkg.globalImageMatchingSets(inp, [c for c, _ in sets], ns, [k for _, k in sets], seed=0)
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
