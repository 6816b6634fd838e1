"""featureMatchingPairwise + imageMatching in one call (aps_pairwise_image_matching[_sets]) against the two-call chains
at the same seed: featureMatchingPairwiseSets -> imageMatchingSets, and featureMatchingPairwise -> imageMatching set by
set (and the one-set fused entry).  Candidate pairs, correspondence offsets, n_inliers, accepted, draws_used, the bits
of the models and their inverses, allMatches, numMatches and tforms must be identical, and return_matches must give
featureMatchingPairwiseSets' lists with their metric.  Also every matching method, subset views, ORB sets, launch
counts that do not depend on the number of sets, more than 65535 candidate pairs, lists with more rows than there are
descriptor rows, and the MEX gateway."""
import numpy as np
import pytest

from test_gpu_global_image_matching import _same_cells, _same_result, make_set

pytestmark = pytest.mark.gpu
PARAMS = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.8, "useMATLABFeatureMatch": 0,
          "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}
METHODS = {"Exhaustive": {}, "subsetpdist2": {"Matchingmethod": "Approximate", "ApproxFloatNNMethod": "subsetpdist2"},
           "kdtree": {"Matchingmethod": "Approximate", "ApproxFloatNNMethod": "kdtree"},
           "pca2nn": {"Matchingmethod": "Approximate", "ApproxFloatNNMethod": "pca2nn"}}


def _same_lists(got, ref, n):
    (gm, gd), (rm, rd) = got, ref
    _same_cells(gm, rm, n)
    for i in range(n):
        for j in range(n):
            assert (gd[i][j] is None) == (rd[i][j] is None), (i, j)
            if gd[i][j] is not None:
                assert np.array_equal(gd[i][j], rd[i][j]), (i, j)


def check_against_chains(aps, inp, cells, kps, seed=3, single=None):
    """the fused call against both chains; single: sets also compared with the one-set chain (default all).
    Returns (accepted pairs, candidate pairs)."""
    ns = [len(c) for c in cells]
    got, lists = aps.pairwiseImageMatchingSets(inp, cells, ns, kps, seed=seed, return_matches=True)
    glast = aps.pairwiseImageMatchingSets.last
    matches = aps.featureMatchingPairwiseSets(inp, cells, ns, return_metric=True)
    ref = aps.imageMatchingSets(inp, ns, kps, [m for m, _ in matches], seed=seed)
    rlast = aps.imageMatchingSets.last
    for b, n in enumerate(ns):
        _same_lists(lists[b], matches[b], n)
        _same_result(got[b], glast[b], ref[b], rlast[b], n)
    for b in (range(len(ns)) if single is None else single):
        mb = aps.featureMatchingPairwise(inp, cells[b], ns[b], return_metric=True)
        r1 = aps.imageMatching(inp, ns[b], kps[b], mb[0], seed=seed)
        _same_result(got[b], glast[b], r1, aps.imageMatching.last if glast[b]["pairs_lin"].size else {}, ns[b])
        g1, m1 = aps.pairwiseImageMatching(inp, cells[b], ns[b], kps[b], seed=seed, return_matches=True)
        _same_result(g1, aps.pairwiseImageMatching.last, r1, glast[b], ns[b])
        _same_lists(m1, mb, ns[b])
    acc = sum(int(l["accepted"].sum()) for l in glast)
    return acc, sum(l["pairs_lin"].size for l in glast)


@pytest.mark.parametrize("method", list(METHODS))
def test_mixed_batch_equals_both_chains(aps, method):
    """sets on the exact engine and sets on the tensor engine (2048 rows per image), a set without descriptors, a
    one-image set and images without descriptors"""
    rng = np.random.default_rng(21)
    shapes = [(4, 300, ()), (3, 2048, ()), (2, 200, (0, 1)), (1, 400, ()), (5, 250, (2,)), (3, 2048, (1,)),
              (3, 150, ())]
    cells, kps = [], []
    for n, kp, empty in shapes:
        c, k = make_set(aps, rng, n, kp, empty=empty)
        cells.append(c), kps.append(k)
    acc, cand = check_against_chains(aps, dict(PARAMS, **METHODS[method]), cells, kps)
    assert 0 < acc < cand, (acc, cand)


def test_subset_views_equal_both_chains(aps):
    """'subsetpdist2' with apsSubset below some images' rows: virtual subset images keyed by the image's index in its
    own set"""
    rng = np.random.default_rng(22)
    cells, kps = [], []
    for n, kp, empty in ((4, 600, ()), (3, 300, ()), (5, 500, (1,))):
        c, k = make_set(aps, rng, n, kp, empty=empty, share=0.5)
        cells.append(c), kps.append(k)
    inp = dict(PARAMS, apsSubset=400, apsSeed=9, **METHODS["subsetpdist2"])
    acc, cand = check_against_chains(aps, inp, cells, kps)
    assert 0 < acc < cand, (acc, cand)


def test_orb_sets_equal_both_chains(aps):
    rng = np.random.default_rng(23)
    cells, kps = [], []
    for n, kp, empty in ((4, 400, ()), (3, 300, (2,)), (1, 100, ()), (5, 500, ())):
        c, k = make_set(aps, rng, n, kp, kind="orb", empty=empty)
        cells.append(c), kps.append(k)
    acc, cand = check_against_chains(aps, dict(PARAMS, Matchingthreshold=40), cells, kps)
    assert 0 < acc < cand, (acc, cand)


@pytest.mark.parametrize("shape", [(6, 2048, (3,)), (30, 4096, ())], ids=["C1", "C5-ring"])
def test_single_c1_and_c5_ring_shaped_sets(aps, shape):
    n, kp, empty = shape
    cells, kps = make_set(aps, np.random.default_rng(24), n, kp, empty=empty)
    acc, cand = check_against_chains(aps, PARAMS, [cells], [kps], seed=7)
    assert 0 < acc < cand, (acc, cand)


def test_launch_count_does_not_depend_on_the_number_of_sets(aps):
    L = aps._lib.lib()
    counts = []
    for B in (2, 200):
        rng = np.random.default_rng(25)
        cells, kps = zip(*[make_set(aps, rng, 4, 120) for _ in range(B)])
        aps.pairwiseImageMatchingSets(PARAMS, list(cells), [4] * B, list(kps))
        c0 = L.aps_launch_count()
        aps.pairwiseImageMatchingSets(PARAMS, list(cells), [4] * B, list(kps))
        counts.append(L.aps_launch_count() - c0)
    assert counts[0] == counts[1], counts


def shared_set(aps, rng, n, kp, random_kp=(), D=128):
    """n images that all hold noisy copies of the same kp rows, so every pair matches most rows; the keypoints of
    every image are a mild homography of one set of keypoints, except those of the images in random_kp"""
    base = np.abs(rng.standard_normal((kp, D))) / 11.0
    bkp = rng.uniform(0.0, 2000.0, (kp, 2))
    cells, kps = [], []
    for i in range(n):
        cells.append(aps.synth._sift_quantise(base + rng.normal(0.0, 0.002, (kp, D))))
        if i in random_kp:
            kps.append(rng.uniform(0.0, 2000.0, (kp, 2)))
            continue
        H = np.eye(3) + rng.normal(0.0, 1.0, (3, 3)) * np.array([[0.05, 0.05, 60.0], [0.05, 0.05, 60.0],
                                                                  [2e-5, 2e-5, 0.0]])
        q = np.c_[bkp, np.ones(kp)] @ H.T
        kps.append(q[:, :2] / q[:, 2:3] + rng.normal(0.0, 0.5, (kp, 2)))
    return cells, kps


def test_more_than_65535_candidate_pairs(aps):
    """11000 sets of 4 images that all share their rows (6 candidate pairs each, 66000 in all, 44000 images): the
    RANSAC runs in two chunks.  Every other set has one image with random keypoints."""
    rng = np.random.default_rng(26)
    B = 11000
    cells, kps = zip(*[shared_set(aps, rng, 4, 16, random_kp=(b % 4,) if b % 2 else ()) for b in range(B)])
    inp = dict(PARAMS, maxIter=4)
    acc, cand = check_against_chains(aps, inp, list(cells), list(kps), seed=5, single=[0, 1, 10922, 10923, B - 1])
    assert cand > 65535 and 0 < acc < cand, (acc, cand)


def test_lists_with_more_rows_than_descriptor_rows(aps):
    """6 images that share their rows: the lists hold far more rows than the F descriptor rows of the set (a query row
    matches once in every pair of its image).  One image's keypoints are random, so its pairs fail RANSAC."""
    n, kp = 6, 400
    cells, kps = shared_set(aps, np.random.default_rng(27), n, kp, random_kp=(4,))
    acc, cand = check_against_chains(aps, PARAMS, [cells], [kps])
    rows = int(aps.pairwiseImageMatchingSets.last[0]["pt_ptr"][-1])
    assert rows > n * kp, rows
    assert 0 < acc < cand, (acc, cand)


def test_gateway_real_call_equals_host_mirror(tmp_path):
    import test_mex_gateways as tg

    pkg = __import__("__graft_entry__").load_package()
    rng = np.random.default_rng(28)
    sets = [make_set(pkg, rng, n, kp, empty=e) for n, kp, e in ((4, 300, ()), (1, 100, ()), (3, 700, (1,)))]
    ns = [len(c) for c, _ in sets]
    mats = []
    for c, k in sets:
        mats += [(0, np.asarray(d, np.float32).reshape(-1, 128)) for d in c]
        mats += [(2, np.asarray(x, np.float64).reshape(-1, 2)) for x in k]
    inp = dict(PARAMS, mBrownLowe=3)
    outs = tg._run_gate("gate_pimatch", mats, [len(ns)] + ns + [1.5, 0.8, 0, 3, 5.5, 99.9, 500, 0], tmp_path)
    ref = pkg.pairwiseImageMatchingSets(inp, [c for c, _ in sets], ns, [k for _, k in sets], seed=0)
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
