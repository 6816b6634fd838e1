"""Device input (the *_dev entries): the one-call matching and image matching verbs fed with CUDA tensors against the
same verbs fed with the same data on the host (.cpu().numpy()).  Every output must be bit-identical: putative lists and
metric, candidate pairs, correspondence offsets, n_inliers, accepted, draws_used, the bits of the models and their
inverses, allMatches, numMatches and tforms.  Covers tensor-path and exact-engine float sets, ORB sets, integer SIFT in
uint8 tensors taken as float, empty images and empty sets, every pairwise method, float32 and float64 keypoints,
C1- and C5-ring-shaped sets, a producer on another stream, launch counts, pointer checks and the one-set forms."""
import ctypes as C

import numpy as np
import pytest

from test_gpu_global_image_matching import _same_cells, _same_result, make_set

pytestmark = pytest.mark.gpu
GLOBAL = {"k": 4, "Ratiothreshold": 0.8, "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500,
          "mBrownLowe": 6}
PAIRWISE = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.8, "useMATLABFeatureMatch": 0,
            "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}
METHODS = {"Exhaustive": {}, "subsetpdist2": {"Matchingmethod": "Approximate", "ApproxFloatNNMethod": "subsetpdist2"},
           "kdtree": {"Matchingmethod": "Approximate", "ApproxFloatNNMethod": "kdtree"},
           "pca2nn": {"Matchingmethod": "Approximate", "ApproxFloatNNMethod": "pca2nn"}}


def _tensors(aps, cells, kps, kind, kp_dtype):
    """host cells / keypoints of make_set -> (descriptor tensors, keypoint tensors) on cuda:0"""
    import torch

    d, k = [], []
    for c, kp in zip(cells, kps):
        a = c.Features if isinstance(c, aps.binaryFeatures) else np.asarray(c)
        if kind == "u8":
            a = a.astype(np.uint8)         # integer SIFT in [0, 255], as vl_SIFT returns it
        d.append(torch.from_numpy(np.ascontiguousarray(a)).cuda())
        k.append(torch.from_numpy(np.ascontiguousarray(kp)).to(kp_dtype).cuda())
    return d, k


def _host(aps, dsets, ksets, binary):
    """the device data as a host caller would pass it"""
    h = [[aps.binaryFeatures(t.cpu().numpy()) if binary else t.cpu().numpy() for t in ds] for ds in dsets]
    return h, [[t.cpu().numpy() for t in ks] for ks in ksets]


def _pairwise_lists(got, ref, n):
    (gm, gd), (rm, rd) = got, ref
    _same_cells(gm, rm, n)
    for i in range(n):
        for j in range(n):
            assert (gd[i][j] is None) == (rd[i][j] is None), (i, j)
            if gd[i][j] is not None:
                assert np.array_equal(gd[i][j], rd[i][j]), (i, j)


def _sets(aps, rng, shapes, kind="sift", kp_dtype=None):
    import torch

    binary = kind == "orb"
    dsets, ksets = [], []
    for n, kp, empty in shapes:
        c, k = make_set(aps, rng, n, kp, kind="orb" if binary else "sift", empty=empty)
        d, kt = _tensors(aps, c, k, kind, kp_dtype or torch.float64)
        dsets.append(d), ksets.append(kt)
    return dsets, ksets, binary


def check_global(aps, inp, dsets, ksets, binary, seed=3, single=(0,)):
    ns = [len(d) for d in dsets]
    hd, hk = _host(aps, dsets, ksets, binary)
    got, glists = aps.globalImageMatchingSetsDevice(inp, dsets, ns, ksets, seed=seed, return_matches=True,
                                                    isBinary=binary)
    glast = aps.globalImageMatchingSetsDevice.last
    ref, rlists = aps.globalImageMatchingSets(inp, hd, ns, hk, seed=seed, return_matches=True)
    rlast = aps.globalImageMatchingSets.last
    lists = aps.featureMatchingGlobalSetsDevice(inp, dsets, ns, isBinary=binary)
    for b, n in enumerate(ns):
        _same_cells(glists[b], rlists[b], n)
        _same_cells(lists[b], rlists[b], n)
        _same_result(got[b], glast[b], ref[b], rlast[b], n)
    for b in single:
        g1, m1 = aps.globalImageMatchingDevice(inp, dsets[b], ns[b], ksets[b], seed=seed, return_matches=True,
                                               isBinary=binary)
        _same_result(g1, aps.globalImageMatchingDevice.last, ref[b], rlast[b], ns[b])
        _same_cells(m1, rlists[b], ns[b])
    return sum(int(l["accepted"].sum()) for l in glast)


def check_pairwise(aps, inp, dsets, ksets, binary, seed=3, single=(0,)):
    ns = [len(d) for d in dsets]
    hd, hk = _host(aps, dsets, ksets, binary)
    got, glists = aps.pairwiseImageMatchingSetsDevice(inp, dsets, ns, ksets, seed=seed, return_matches=True,
                                                      isBinary=binary)
    glast = aps.pairwiseImageMatchingSetsDevice.last
    ref, rlists = aps.pairwiseImageMatchingSets(inp, hd, ns, hk, seed=seed, return_matches=True)
    rlast = aps.pairwiseImageMatchingSets.last
    lists = aps.featureMatchingPairwiseSetsDevice(inp, dsets, ns, return_metric=True, isBinary=binary)
    for b, n in enumerate(ns):
        _pairwise_lists(glists[b], rlists[b], n)
        _pairwise_lists(lists[b], rlists[b], n)
        _same_result(got[b], glast[b], ref[b], rlast[b], n)
    for b in single:
        g1, m1 = aps.pairwiseImageMatchingDevice(inp, dsets[b], ns[b], ksets[b], seed=seed, return_matches=True,
                                                 isBinary=binary)
        _same_result(g1, aps.pairwiseImageMatchingDevice.last, ref[b], rlast[b], ns[b])
        _pairwise_lists(m1, rlists[b], ns[b])
        one = aps.featureMatchingPairwiseDevice(inp, dsets[b], ns[b], return_metric=True, isBinary=binary)
        _pairwise_lists(one, aps.featureMatchingPairwise(inp, hd[b], ns[b], return_metric=True), ns[b])
    return sum(int(l["accepted"].sum()) for l in glast)


# tensor-path sets (>= 2048 rows per image) after exact-engine sets, a set without descriptors, a one-image set and
# images without descriptors
MIXED = [(4, 300, ()), (3, 2048, ()), (2, 200, (0, 1)), (1, 400, ()), (5, 250, (2,)), (3, 2048, (1,))]


@pytest.mark.parametrize("kp64", [True, False], ids=["kp-f64", "kp-f32"])
@pytest.mark.parametrize("kind", ["sift", "u8", "orb"])
def test_global_sets_device_equals_host(aps, kind, kp64):
    import torch

    shapes = MIXED if kind != "orb" else [(4, 400, ()), (3, 300, (2,)), (1, 100, ()), (2, 50, (0, 1))]
    dsets, ksets, binary = _sets(aps, np.random.default_rng(31), shapes, kind,
                                 torch.float64 if kp64 else torch.float32)
    inp = dict(GLOBAL, BFMatch=1) if binary else GLOBAL
    assert check_global(aps, inp, dsets, ksets, binary, single=(0, 1, 2)) > 0


@pytest.mark.parametrize("method", list(METHODS))
def test_pairwise_sets_device_equals_host(aps, method):
    import torch

    dsets, ksets, binary = _sets(aps, np.random.default_rng(32), MIXED, "sift", torch.float32)
    assert check_pairwise(aps, dict(PAIRWISE, **METHODS[method]), dsets, ksets, binary, single=(0, 1)) > 0


def test_pairwise_subset_views_and_u8_and_orb(aps):
    rng = np.random.default_rng(33)
    dsets, ksets, binary = _sets(aps, rng, [(4, 600, ()), (3, 300, ()), (5, 500, (1,))], "u8")
    inp = dict(PAIRWISE, apsSubset=400, apsSeed=9, **METHODS["subsetpdist2"])
    assert check_pairwise(aps, inp, dsets, ksets, binary, single=(0, 2)) > 0
    dsets, ksets, binary = _sets(aps, rng, [(4, 400, ()), (3, 300, (2,)), (1, 100, ())], "orb")
    assert check_pairwise(aps, dict(PAIRWISE, Matchingthreshold=40), dsets, ksets, binary) > 0


def test_all_sets_empty(aps):
    import torch

    e = torch.zeros((0, 128), device="cuda")
    k = torch.zeros((0, 2), device="cuda", dtype=torch.float64)
    assert check_global(aps, GLOBAL, [[e, e], [e]], [[k, k], [k]], False) == 0
    assert check_pairwise(aps, PAIRWISE, [[e, e], [e]], [[k, k], [k]], False) == 0


@pytest.mark.parametrize("shape", [(6, 2048, (3,)), (30, 4096, ())], ids=["C1", "C5-ring"])
def test_c1_and_c5_ring_shaped_sets(aps, shape):
    import torch

    dsets, ksets, binary = _sets(aps, np.random.default_rng(34), [shape], "sift", torch.float32)
    assert check_global(aps, GLOBAL, dsets, ksets, binary, seed=7) > 0
    assert check_pairwise(aps, PAIRWISE, dsets, ksets, binary, seed=7) > 0


def test_producer_on_another_stream(aps):
    """descriptors and keypoints written by torch on a side stream right before the call, without a host
    synchronisation: the call's stream waits for the producer's event"""
    import torch

    dsets, ksets, _ = _sets(aps, np.random.default_rng(35), [(4, 2048, ()), (3, 700, ())], "sift")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        w = torch.randn(8192, 8192, device="cuda")
        for _ in range(4):
            w = torch.tanh(w @ w)             # a long producer: the copies below come after it on `side`
        zero = (w.sum() * 0.0).nan_to_num()
        prod_d = [[torch.empty_like(t).copy_(t + zero) for t in ds] for ds in dsets]
        prod_k = [[torch.empty_like(t).copy_(t + zero.double()) for t in ks] for ks in ksets]
        got = aps.globalImageMatchingSetsDevice(GLOBAL, prod_d, [4, 3], prod_k, seed=5)
        glast = aps.globalImageMatchingSetsDevice.last
    torch.cuda.synchronize()
    hd, hk = _host(aps, dsets, ksets, False)
    ref = aps.globalImageMatchingSets(GLOBAL, hd, [4, 3], hk, seed=5)
    for b, n in enumerate([4, 3]):
        _same_result(got[b], glast[b], ref[b], aps.globalImageMatchingSets.last[b], n)
    assert sum(int(l["accepted"].sum()) for l in glast) > 0


def test_producer_on_the_default_stream(aps):
    """the motivating case: an extractor writes CUDA tensors on torch's default stream and the caller calls the verb
    right away, without a synchronisation.  torch reports that stream as handle 0; it is handed over as
    cudaStreamLegacy, so the context's non-blocking stream waits for the producer"""
    import torch

    assert torch.cuda.current_stream().cuda_stream == 0
    assert aps.host._producer_stream(torch.device("cuda", 0)).value == aps.host.CUDA_STREAM_LEGACY
    dsets, ksets, _ = _sets(aps, np.random.default_rng(37), [(4, 2048, ()), (3, 700, ())], "sift", torch.float32)
    hd, hk = _host(aps, dsets, ksets, False)
    for verb, inp in (("global", GLOBAL), ("pairwise", PAIRWISE)):
        torch.cuda.synchronize()
        w = torch.randn(8192, 8192, device="cuda")
        for _ in range(4):
            w = torch.tanh(w @ w)             # a long producer: the tensors below are written after it
        zero = (w.sum() * 0.0).nan_to_num()
        prod_d = [[t + zero for t in ds] for ds in dsets]
        prod_k = [[t + zero for t in ks] for ks in ksets]
        got = getattr(aps, f"{verb}ImageMatchingSetsDevice")(inp, prod_d, [4, 3], prod_k, seed=5)
        glast = getattr(aps, f"{verb}ImageMatchingSetsDevice").last
        one = getattr(aps, f"featureMatching{verb.capitalize()}SetsDevice")(inp, [[t + zero for t in dsets[1]]], [3])
        ref = getattr(aps, f"{verb}ImageMatchingSets")(inp, hd, [4, 3], hk, seed=5)
        rlast = getattr(aps, f"{verb}ImageMatchingSets").last
        for b, n in enumerate([4, 3]):
            _same_result(got[b], glast[b], ref[b], rlast[b], n)
        _same_cells(one[0], getattr(aps, f"featureMatching{verb.capitalize()}Sets")(inp, [hd[1]], [3])[0], 3)
        assert sum(int(l["accepted"].sum()) for l in glast) > 0, verb


def test_launches_no_more_than_host_and_independent_of_sets(aps):
    """float64 keypoints: the same launches as the host-input calls, for one set and for many.  float32 keypoints: one
    launch more, the widening kernel -- a deliberate exception to 'never more launches than the host-input call', since
    the host route widens on the host before its upload.  The context statistics are the host call's too."""
    import torch

    L = aps._lib.lib()
    ctx = aps._lib.default_context()

    def launches(fn):
        fn()
        c0 = L.aps_launch_count()
        fn()
        return L.aps_launch_count() - c0

    def stats(fn):
        fn()
        return ctx.last_stats(), ctx.pairwise_stats()

    for B in (1, 2, 100):
        rng = np.random.default_rng(36)
        dsets, ksets, _ = _sets(aps, rng, [(4, 120, ())] * B, "sift")
        k32 = [[t.float() for t in ks] for ks in ksets]
        hd, hk = _host(aps, dsets, ksets, False)
        ns = [4] * B
        for verb, inp in (("global", GLOBAL), ("pairwise", PAIRWISE)):
            host = getattr(aps, f"{verb}ImageMatchingSets")
            dev = getattr(aps, f"{verb}ImageMatchingSetsDevice")
            n_host = launches(lambda: host(inp, hd, ns, hk))
            assert launches(lambda: dev(inp, dsets, ns, ksets)) == n_host, (verb, B)
            assert launches(lambda: dev(inp, dsets, ns, k32)) == n_host + 1, (verb, B)
        for verb, inp in (("Global", GLOBAL), ("Pairwise", PAIRWISE)):
            host = lambda: getattr(aps, f"featureMatching{verb}Sets")(inp, hd, ns)              # noqa: E731
            dev = lambda: getattr(aps, f"featureMatching{verb}SetsDevice")(inp, dsets, ns)     # noqa: E731
            assert launches(dev) == launches(host), (verb, B)
            assert stats(dev) == stats(host), (verb, B)
        if B == 1:
            one = lambda: aps.featureMatchingPairwise(PAIRWISE, hd[0], 4)                       # noqa: E731
            one_dev = lambda: aps.featureMatchingPairwiseDevice(PAIRWISE, dsets[0], 4)          # noqa: E731
            assert launches(one_dev) == launches(one)
            assert stats(one_dev) == stats(one)
        if B == 2:
            first = launches(lambda: aps.globalImageMatchingSetsDevice(GLOBAL, dsets, ns, ksets))
    assert launches(lambda: aps.globalImageMatchingSetsDevice(GLOBAL, dsets, ns, ksets)) == first


def test_host_and_null_pointers_are_refused(aps):
    import torch

    L = aps._lib.lib()
    ctx = aps._lib.default_context()
    host = np.zeros((64, 128), np.float32)
    kp_host = np.zeros((64, 2))
    dev = torch.zeros((64, 128), device="cuda")
    kp_dev = torch.zeros((64, 2), device="cuda", dtype=torch.float64)
    si = (C.c_int * 1)(2)
    cnt = (C.c_int64 * 2)(32, 32)
    for d in (host.ctypes.data, None):
        outs = (C.c_void_p * 1)()
        assert L.aps_feature_matching_global_sets_dev(ctx.handle, 1, si, d, cnt, 128, 0, 4, 0.8, 0, 0, None, outs) == 1
        assert L.aps_feature_matching_pairwise_sets_dev(ctx.handle, 1, si, d, cnt, 128, 0, 1.5, 0.8, 0, 12000, 0, None,
                                                        outs) == 1
    h = C.c_void_p()
    for d, k in ((host.ctypes.data, kp_dev.data_ptr()), (dev.data_ptr(), kp_host.ctypes.data),
                 (None, kp_dev.data_ptr()), (dev.data_ptr(), None)):
        assert L.aps_global_image_matching_sets_dev(ctx.handle, 1, si, d, cnt, 128, 0, 4, 0.8, 0, 0, k, 0, 6, 5.5,
                                                    99.9, 500, 0, 0, None, C.byref(h)) == 1
        assert L.aps_pairwise_image_matching_sets_dev(ctx.handle, 1, si, d, cnt, 128, 0, 1.5, 0.8, 0, 12000, 0, k, 0, 6,
                                                      5.5, 99.9, 500, 0, 0, None, C.byref(h)) == 1
    with pytest.raises(TypeError):
        aps.featureMatchingGlobalSetsDevice(GLOBAL, [[torch.zeros((4, 128)), torch.zeros((4, 128))]], [2])
