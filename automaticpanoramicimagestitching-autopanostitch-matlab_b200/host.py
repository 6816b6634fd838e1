"""Host-side mirror of the reference's MATLAB interface for the feature-matching path.

Same function names, argument meaning and error behaviour as the reference (PP/ = "Procedural
Program/"), so the parity tests read like the reference's call sites:

  featureMatchingGlobal(input, allDescriptors, numImg)        PP/featureMatching/featureMatchingGlobal.m:1
  featureMatchingPairwise(input, allDescriptors, numImg)      PP/featureMatching/featureMatchingPairwise.m:1
  matchFeaturesScratch(F1, F2, Method=..., MatchThreshold=..) PP/featureMatching/matchFeaturesScratch.m:1
  flann_knn_win(train[, query], k[, method, trees, checks])   PP/mex/flann_knn.cpp:118-253
  nearest2HammingExhaustiveMEX(A, B) / ...OMPMEX(A, B)        PP/mex/nearest2HammingExhaustive{,OMP}MEX.cpp
  nearest2SSDExhaustive(A, B)                                 PP/featureMatching/matchFeaturesScratch.m:322-366
  selectImagePartners(matchesAll, m)                          PP/imageMatching/imageMatching.m:75-100

MATLAB is not available in this image, so this mirror is Python; it only marshals arguments into
the C ABI (include/apsmatch.h).  All arithmetic runs in libapsmatch.so on the GPU; nothing here
computes a distance.  `input` may be a dict or any object with the reference's field names.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from ._lib import APS_COL_MAJOR, APS_F32, APS_ROW_MAJOR, APS_U8, ApsError, check, default_context, lib


class binaryFeatures:
    """Stand-in for MATLAB's binaryFeatures object (featureMatchingGlobal.m:56-75, matchFeaturesScratch.m:259-262): packed uint8 rows in `.Features`."""

    def __init__(self, features):
        f = np.asarray(features)
        if f.dtype != np.uint8 or f.ndim != 2:
            raise TypeError("binaryFeatures expects an [N x nbytes] uint8 matrix")
        self.Features = f
        self.NumFeatures = f.shape[0]


def _field(inp, name, default=None, required=False):
    if isinstance(inp, dict):
        if name in inp:
            return inp[name]
    elif hasattr(inp, name):
        return getattr(inp, name)
    if required:
        raise KeyError(f"input.{name} is required")
    return default


def _as_matrix(a, dtype):
    """numpy array -> (buffer, layout).  Fortran-ordered arrays go through as MATLAB column-major."""
    a = np.asarray(a)
    if a.ndim != 2:
        raise ApsError(2, "flann_knn:type", "descriptors must be 2D")
    if a.dtype != dtype:
        a = a.astype(dtype)
    if a.flags.c_contiguous:
        return a, APS_ROW_MAJOR
    if a.flags.f_contiguous:
        return a, APS_COL_MAJOR
    return np.ascontiguousarray(a), APS_ROW_MAJOR


def _ptr(a):
    return C.c_void_p(a.ctypes.data) if a.size else C.c_void_p(0)


def _cells_from_matchlist(h, n, want_metric=False):
    L = lib()
    total = L.aps_matchlist_total(h)
    pp = np.ctypeslib.as_array(L.aps_matchlist_pair_ptr(h), shape=(n * n + 1,)).copy()
    rows = (np.ctypeslib.as_array(L.aps_matchlist_rows(h), shape=(total, 2)).copy() if total
            else np.zeros((0, 2), np.uint32))
    mp = L.aps_matchlist_metric(h)
    metric = np.ctypeslib.as_array(mp, shape=(total,)).copy() if (want_metric and total and mp) else None
    nothing = np.zeros((0, 0))
    matches = [[nothing] * n for _ in range(n)]  # cell(numImg): every entry []
    metrics = [[None] * n for _ in range(n)]
    # double, [M x 2] (featureMatchingGlobal.m:155-159): one conversion, then views per cell
    rows_f = rows.astype(np.float64)
    filled = np.flatnonzero(np.diff(pp) > 0)
    for c in filled.tolist():
        i, j = c % n, c // n
        if i < j:
            matches[i][j] = rows_f[pp[c]:pp[c + 1]]
            if metric is not None:
                metrics[i][j] = metric[pp[c]:pp[c + 1]]
    return matches, metrics, pp, rows


def _describe(allDescriptors, numImg):
    """Shared front end: detect binary vs float, per-image matrices, counts (featureMatchingGlobal.m:48-63)."""
    n = int(numImg)
    cells = list(allDescriptors) if allDescriptors is not None else []
    if len(cells) < n:
        cells = cells + [None] * (n - len(cells))

    def is_empty(x):
        if x is None:
            return True
        if isinstance(x, binaryFeatures):
            return x.NumFeatures == 0
        return np.asarray(x).size == 0

    first = next((x for x in cells[:n] if not is_empty(x)), None)
    if first is None:
        return n, None, [], [], 0, False
    is_binary = isinstance(first, binaryFeatures)
    mats, counts = [], []
    D = None
    for x in cells[:n]:
        if is_empty(x):
            mats.append(None)
            counts.append(0)
            continue
        m = x.Features if isinstance(x, binaryFeatures) else np.asarray(x)
        if is_binary:
            if m.dtype != np.uint8:
                raise ApsError(2, "flann_knn:type", "binary descriptors must be uint8")
        elif m.dtype not in (np.float32, np.float64) and not np.issubdtype(m.dtype, np.integer):
            raise ApsError(2, "flann_knn:type", "Descriptors must be single (float) or uint8 (binary)")
        m, _ = _as_matrix(m, np.uint8 if is_binary else np.float32)  # single(allDesc), :81
        if D is None:
            D = m.shape[1]
        elif m.shape[1] != D:
            raise ApsError(4, "flann_knn:dim", "all descriptor matrices must have the same number of columns")
        mats.append(m)
        counts.append(m.shape[0])
    return n, first, mats, counts, D, is_binary


def _desc_args(mats, counts):
    n = len(counts)
    layouts = {(_as_matrix(m, m.dtype)[1]) for m in mats if m is not None}
    layout = APS_ROW_MAJOR
    if layouts == {APS_COL_MAJOR}:
        layout = APS_COL_MAJOR
    elif len(layouts) > 1:
        mats = [None if m is None else np.ascontiguousarray(m) for m in mats]
    ptrs = (C.c_void_p * max(n, 1))()
    for i, m in enumerate(mats):
        ptrs[i] = m.ctypes.data if m is not None and m.size else None
    cnt = (C.c_int64 * max(n, 1))(*counts) if n else (C.c_int64 * 1)()
    return ptrs, cnt, layout, mats


def _aps_gpus(input, ctx):
    """input.apsGPUs: GPUs to spread the call over, 1-based like MATLAB's gpuDevice.  Returns (group or None, ctx):
    a DeviceGroup when more than one GPU is listed; one GPU -> that GPU's default context (unless ctx is given)."""
    gpus = _field(input, "apsGPUs", None)
    if gpus is None:
        return None, ctx or default_context()
    g = np.atleast_1d(np.asarray(gpus, dtype=np.float64)).ravel()
    if g.size and (not np.all(np.isfinite(g)) or np.any(g != np.round(g)) or np.any(g < 1)
                   or len(set(g.tolist())) != g.size):
        raise ValueError("input.apsGPUs must list distinct positive integer GPU indices (1-based, as gpuDevice)")
    devices = [int(v) - 1 for v in g]
    if len(devices) > 1:
        if ctx is not None:
            raise ValueError("input.apsGPUs with several GPUs and ctx= are alternative ways to choose the device")
        return _lib.default_group(devices), None
    return None, ctx or default_context(devices[0] if devices else 0)


def featureMatchingGlobal(input, allDescriptors, numImg, ctx=None):
    """matches = featureMatchingGlobal(input, allDescriptors, numImg)   (featureMatchingGlobal.m:1-163)

    Returns an n x n nested list `matches[i][j]` (0-based): [M x 2] float64 index pairs (1-based
    local feature indices, column 0 -> image i, column 1 -> image j) for i < j, empty elsewhere.
    input.apsGPUs (1-based GPU indices) listing several GPUs spreads the call over them (aps_group_feature_matching_global,
    same lists)."""
    group, ctx = _aps_gpus(input, ctx)
    if not (np.isscalar(numImg) and np.isfinite(numImg) and numImg > 0):
        raise ValueError("numImg must be a positive finite scalar")  # arguments block :35-39
    k = int(_field(input, "k", required=True))
    ratio = float(_field(input, "Ratiothreshold", required=True))
    use_bf = bool(_field(input, "BFMatch", 0))
    mutual = bool(int(_field(input, "apsMutual", 0)))   # opt-in cross-check, NOT reference behaviour (include/apsmatch.h)
    n, first, mats, counts, D, is_binary = _describe(allDescriptors, numImg)
    if first is None:
        return [[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)]  # :49-52
    ptrs, cnt, layout, keep = _desc_args(mats, counts)
    h = C.c_void_p()
    if group is not None:
        check(lib().aps_group_feature_matching_global(group.handle, ptrs, cnt, n, int(D), APS_U8 if is_binary else APS_F32,
                                                      layout, k, ratio, int(mutual), C.byref(h)))
        try:
            return _cells_from_matchlist(h, n)[0]
        finally:
            lib().aps_matchlist_free(h)
    if mutual:
        plan = GlobalPlan(ctx, counts, D, is_binary, k)
        try:
            plan.upload(mats)
            plan.prepare()
            plan.knn()
            plan.filter(ratio)
            plan.filter_mutual()
            plan.compact()
            return plan.download()[0]
        finally:
            plan.close()
    check(lib().aps_feature_matching_global(ctx.handle, ptrs, cnt, n, int(D), APS_U8 if is_binary else APS_F32, layout,
                                            k, ratio, int(use_bf), C.byref(h)))
    try:
        matches, _, _, _ = _cells_from_matchlist(h, n)
    finally:
        lib().aps_matchlist_free(h)
    return matches


def featureMatchingGlobalSets(input, allDescriptorsSets, numImgs, ctx=None):
    """matchesSets = featureMatchingGlobalSets(input, allDescriptorsSets, numImgs)

    featureMatchingGlobal over B independent image sets in one call (aps_feature_matching_global_sets): set b is
    allDescriptorsSets[b] with numImgs[b] images.  Returns a list of B nested lists, element b exactly what
    featureMatchingGlobal(input, allDescriptorsSets[b], numImgs[b]) returns (with input.apsMutual too).  All sets share
    one descriptor kind (float or binaryFeatures) and width.  Device groups (input.apsGPUs) are not supported here."""
    if _field(input, "apsGPUs", None) is not None:
        raise ValueError("input.apsGPUs is not supported by featureMatchingGlobalSets; match the sets on one GPU")
    sets = list(allDescriptorsSets) if allDescriptorsSets is not None else []
    nums = list(np.atleast_1d(np.asarray(numImgs, dtype=np.float64)).ravel()) if np.size(numImgs) else []
    if len(nums) != len(sets):
        raise ValueError("numImgs must give one image count per descriptor set")
    for v in nums:
        if not (np.isfinite(v) and v > 0 and v == np.round(v)):
            raise ValueError("every numImgs entry must be a positive integer")  # featureMatchingGlobal.m:35-39
    k = int(_field(input, "k", required=True))
    ratio = float(_field(input, "Ratiothreshold", required=True))
    use_bf = bool(_field(input, "BFMatch", 0))
    mutual = bool(int(_field(input, "apsMutual", 0)))
    ns, all_mats, all_counts = [], [], []
    kind = D = None
    for cells, num in zip(sets, nums):
        n, first, mats, counts, Db, is_binary = _describe(cells, num)
        if first is None:
            mats, counts = [None] * n, [0] * n
        else:
            if kind is not None and is_binary != kind:
                raise ApsError(2, "flann_knn:type", "all descriptor sets must have the same class")
            if D is not None and Db != D:
                raise ApsError(4, "flann_knn:dim", "all descriptor sets must have the same number of columns")
            kind, D = is_binary, Db
        ns.append(n)
        all_mats += mats
        all_counts += counts
    B = len(ns)
    if kind is None:  # every set empty: cell(numImg) each, no device touched (featureMatchingGlobal.m:49-52)
        return [[[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)] for n in ns]
    ptrs, cnt, layout, keep = _desc_args(all_mats, all_counts)
    simg = (C.c_int * max(B, 1))(*ns)
    outs = (C.c_void_p * max(B, 1))()
    ctx = ctx or default_context()
    check(lib().aps_feature_matching_global_sets(ctx.handle, B, simg, ptrs, cnt, int(D),
                                                 APS_U8 if kind else APS_F32, layout, k, ratio, int(use_bf),
                                                 int(mutual), outs))
    result = []
    try:
        for b in range(B):
            result.append(_cells_from_matchlist(outs[b], ns[b])[0])
    finally:
        for b in range(B):
            lib().aps_matchlist_free(outs[b])
    return result


class ApsSemanticsWarning(UserWarning):
    """The call was served with semantics that differ from what the reference's defaults select."""


APS_METHOD = {"exhaustive": 0, "subsetpdist2": 1, "kdtree": 2, "pca2nn": 3}


def _resolve_method(input, method):
    """(Matchingmethod, ApproxFloatNNMethod) -> aps_method (include/apsmatch.h), following matchFeaturesScratch.m:116-163.
    PP/inputs.m:47-49 defaults: useMATLABFeatureMatch=1 (MathWorks matchFeatures, closed source), 'Approximate',
    'subsetpdist2'.  Nothing here may change results silently: the closed-source branch warns; all three
    ApproxFloatNNMethod values are built (include/apsmatch.h, aps_method)."""
    import warnings

    accept = bool(int(_field(input, "apsAcceptScratchSemantics", 0)))
    if int(_field(input, "useMATLABFeatureMatch", 0)) == 1 and not accept:
        warnings.warn("input.useMATLABFeatureMatch=1 selects MathWorks matchFeatures in the reference (closed source); "
                      "this GPU path runs the matchFeaturesScratch semantics (featureMatchingPairwise.m:108-117). "
                      "Set input.apsAcceptScratchSemantics=1 to acknowledge.", ApsSemanticsWarning, stacklevel=3)
    if method == "exhaustive":
        return APS_METHOD["exhaustive"]
    nn = str(_field(input, "ApproxFloatNNMethod", "pca2nn")).lower()     # parser default, matchFeaturesScratch.m:75
    if nn in ("subsetpdist2", "kdtree", "pca2nn"):
        return APS_METHOD[nn]
    raise ValueError("Select a approximate method")                      # :156-157


def featureMatchingGlobalDevice(input, d_pooled, counts, D, is_binary=False, ctx=None):
    """featureMatchingGlobal for descriptors that already live on the device (aps_feature_matching_global_dev):
    d_pooled = device pointer (int) of the pooled ROW-major [sum(counts) x D] matrix, float32 or uint8 -- e.g. a torch
    tensor's data_ptr().  Returns the same n x n nested list."""
    ctx = ctx or default_context()
    n = len(counts)
    cnt = (C.c_int64 * max(n, 1))(*[int(c) for c in counts])
    h = C.c_void_p()
    check(lib().aps_feature_matching_global_dev(ctx.handle, C.c_void_p(int(d_pooled)), cnt, n, int(D),
                                                APS_U8 if is_binary else APS_F32, int(_field(input, "k", required=True)),
                                                float(_field(input, "Ratiothreshold", required=True)),
                                                int(bool(int(_field(input, "apsMutual", 0)))), C.byref(h)))
    try:
        matches, _, _, _ = _cells_from_matchlist(h, n)
    finally:
        lib().aps_matchlist_free(h)
    return matches


def featureMatchingPairwise(input, allDescriptors, numImg, ctx=None, return_metric=False, shard=None, csr=False):
    """matches = featureMatchingPairwise(input, allDescriptors, numImg)  (featureMatchingPairwise.m:1-63)

    Runs getMatches' matchFeaturesScratch branch (:108-117) with Unique=true for every i<j.
    input.useMATLABFeatureMatch=1 (the reference default, PP/inputs.m:47) selects MathWorks' closed-source
    matchFeatures there; here it is served by the matchFeaturesScratch semantics and an ApsSemanticsWarning
    says so (silence it with input.apsAcceptScratchSemantics=1).  Matchingmethod='Approximate' follows
    input.ApproxFloatNNMethod: 'subsetpdist2' (the inputs.m default), 'kdtree' (Euclidean searches) and 'pca2nn' (PCA-48
    + cosine similarity), include/apsmatch.h aps_method.  Binary descriptors always run the exhaustive Hamming search, as
    the reference does (matchFeaturesScratch.m:611).
    shard=(first, stride): compute only every stride-th pair of the column-major pair list (one share
    per GPU rank); cells of other shares come back empty and are merged by `merge_pairwise_shards`.
    csr=True returns the compacted lists as they leave the C ABI: (pair_ptr [n*n+1], rows [M x 2] uint32, metric [M]).
    input.apsGPUs (1-based GPU indices) listing several GPUs spreads the pairs over them in this process
    (aps_group_feature_matching_pairwise, same lists); it cannot be combined with shard=."""
    if shard is not None and _field(input, "apsGPUs", None) is not None:
        raise ValueError("input.apsGPUs and shard= are alternative ways to split the image pairs; pass one of them")
    group, ctx = _aps_gpus(input, ctx)
    if not (np.isscalar(numImg) and np.isfinite(numImg) and numImg > 0):
        raise ValueError("numImg must be a positive finite scalar")
    method = str(_field(input, "Matchingmethod", "Exhaustive")).lower()
    if method not in ("exhaustive", "approximate"):
        raise ValueError(f"Unknown Method: {method}")  # matchFeaturesScratch.m:164-165
    aps_method = _resolve_method(input, method)
    thr = float(_field(input, "Matchingthreshold", required=True))
    ratio = float(_field(input, "Ratiothreshold", required=True))
    n, first, mats, counts, D, is_binary = _describe(allDescriptors, numImg)
    if first is None:
        if csr:
            return np.zeros(n * n + 1, np.int64), np.zeros((0, 2), np.uint32), np.zeros(0)
        m = [[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)]
        return (m, [[None] * n for _ in range(n)]) if return_metric else m
    ptrs, cnt, layout, keep = _desc_args(mats, counts)
    h = C.c_void_p()
    first, stride = shard if shard is not None else (0, 1)
    if group is not None:
        check(lib().aps_group_feature_matching_pairwise(group.handle, ptrs, cnt, n, int(D), APS_U8 if is_binary else APS_F32,
                                                        layout, thr, ratio, aps_method, int(_field(input, "apsSubset", 12000)),
                                                        int(_field(input, "apsSeed", 0)), C.byref(h)))
    elif aps_method != APS_METHOD["exhaustive"] and not is_binary:
        ph = C.c_void_p()
        check(lib().aps_pplan_create(ctx.handle, cnt, n, int(D), APS_F32, C.byref(ph)))
        try:
            check(lib().aps_pplan_set_method(ph, aps_method, int(_field(input, "apsSubset", 12000)),   # 12000: :151
                                             int(_field(input, "apsSeed", 0))))
            check(lib().aps_pplan_upload(ph, ptrs, layout))
            check(lib().aps_pplan_prepare(ph))
            check(lib().aps_pplan_match(ph, thr, ratio, int(first), int(stride), C.byref(h)))
        finally:
            lib().aps_pplan_destroy(ph)
    else:
        check(lib().aps_feature_matching_pairwise_shard(ctx.handle, ptrs, cnt, n, int(D), APS_U8 if is_binary else APS_F32,
                                                        layout, thr, ratio, int(first), int(stride), C.byref(h)))
    try:
        if csr:
            return _csr_from_matchlist(h, n)
        matches, metrics, _, _ = _cells_from_matchlist(h, n, want_metric=True)
    finally:
        lib().aps_matchlist_free(h)
    _fill_upper_cells(matches, n)
    return (matches, metrics) if return_metric else matches


def featureMatchingPairwiseSets(input, allDescriptorsSets, numImgs, ctx=None, return_metric=False):
    """matchesSets = featureMatchingPairwiseSets(input, allDescriptorsSets, numImgs)

    featureMatchingPairwise over B independent image sets in one call (aps_feature_matching_pairwise_sets): set b is
    allDescriptorsSets[b] with numImgs[b] images.  Returns a list of B elements, element b exactly what
    featureMatchingPairwise(input, allDescriptorsSets[b], numImgs[b], return_metric=return_metric) returns.  Reads the
    fields featureMatchingPairwise reads (Matchingmethod, ApproxFloatNNMethod, Matchingthreshold, Ratiothreshold,
    apsSubset, apsSeed) and warns the same way for useMATLABFeatureMatch=1.  All sets share one descriptor kind (float
    or binaryFeatures) and width.  Device groups (input.apsGPUs) are not supported here."""
    if _field(input, "apsGPUs", None) is not None:
        raise ValueError("input.apsGPUs is not supported by featureMatchingPairwiseSets; match the sets on one GPU")
    sets = list(allDescriptorsSets) if allDescriptorsSets is not None else []
    nums = list(np.atleast_1d(np.asarray(numImgs, dtype=np.float64)).ravel()) if np.size(numImgs) else []
    if len(nums) != len(sets):
        raise ValueError("numImgs must give one image count per descriptor set")
    for v in nums:
        if not (np.isfinite(v) and v > 0 and v == np.round(v)):
            raise ValueError("every numImgs entry must be a positive integer")  # featureMatchingPairwise.m arguments
    method = str(_field(input, "Matchingmethod", "Exhaustive")).lower()
    if method not in ("exhaustive", "approximate"):
        raise ValueError(f"Unknown Method: {method}")  # matchFeaturesScratch.m:164-165
    aps_method = _resolve_method(input, method)
    thr = float(_field(input, "Matchingthreshold", required=True))
    ratio = float(_field(input, "Ratiothreshold", required=True))
    ns, empty, all_mats, all_counts = [], [], [], []
    kind = D = None
    for cells, num in zip(sets, nums):
        n, first, mats, counts, Db, is_binary = _describe(cells, num)
        if first is None:
            mats, counts = [None] * n, [0] * n
        else:
            if kind is not None and is_binary != kind:
                raise ApsError(2, "flann_knn:type", "all descriptor sets must have the same class")
            if D is not None and Db != D:
                raise ApsError(4, "flann_knn:dim", "all descriptor sets must have the same number of columns")
            kind, D = is_binary, Db
        ns.append(n)
        empty.append(first is None)
        all_mats += mats
        all_counts += counts

    def empty_cells(n):   # featureMatchingPairwise on a set without descriptors: cell(numImg), no device touched
        m = [[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)]
        return (m, [[None] * n for _ in range(n)]) if return_metric else m

    B = len(ns)
    if kind is None:
        return [empty_cells(n) for n in ns]
    ptrs, cnt, layout, keep = _desc_args(all_mats, all_counts)
    simg = (C.c_int * max(B, 1))(*ns)
    outs = (C.c_void_p * max(B, 1))()
    ctx = ctx or default_context()
    check(lib().aps_feature_matching_pairwise_sets(ctx.handle, B, simg, ptrs, cnt, int(D), APS_U8 if kind else APS_F32,
                                                   layout, thr, ratio, aps_method, int(_field(input, "apsSubset", 12000)),
                                                   int(_field(input, "apsSeed", 0)), outs))
    result = []
    try:
        for b in range(B):
            if empty[b]:
                result.append(empty_cells(ns[b]))
                continue
            matches, metrics, _, _ = _cells_from_matchlist(outs[b], ns[b], want_metric=True)
            _fill_upper_cells(matches, ns[b])
            result.append((matches, metrics) if return_metric else matches)
    finally:
        for b in range(B):
            lib().aps_matchlist_free(outs[b])
    return result


def _fill_upper_cells(matches, n):
    """featureMatchingPairwise fills EVERY upper-triangle cell (possibly 0 x 2), featureMatchingPairwise.m:62."""
    empty = np.zeros((0, 2))
    for j in range(n):
        for i in range(j):
            if matches[i][j].size == 0:
                matches[i][j] = empty


def merge_pairwise_csr(n, counts, rows_all, metric_all=None):
    """Merges the exchanged per-rank CSR lists (multigpu.exchange_pairwise_lists): pair o of the column-major pair
    list was computed by rank o % world; its rows sit in that rank's buffer at the offset its own counts imply."""
    world = counts.shape[0]
    offs = np.concatenate([np.zeros((world, 1), np.int64), np.cumsum(counts, axis=1)], axis=1)
    out = [[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)]
    rows_f = rows_all.astype(np.float64)
    o = 0
    for j in range(n):
        for i in range(j):
            r, c = o % world, i + j * n
            out[i][j] = rows_f[r, offs[r, c]:offs[r, c + 1]]
            o += 1
    _fill_upper_cells(out, n)
    return out


def merge_pairwise_shards(shards):
    """Merges the per-rank results of featureMatchingPairwise(..., shard=(r, world)): every pair was computed
    by exactly one rank, so the merge takes each cell from the rank that owns it (ordinal % world)."""
    world = len(shards)
    n = len(shards[0])
    out = [[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)]
    o = 0
    for j in range(n):
        for i in range(j):
            out[i][j] = shards[o % world][i][j]
            o += 1
    return out


def matchFeaturesScratch(F1, F2, Method="Exhaustive", MatchThreshold=3.5, MaxRatio=0.6, Unique=True, ctx=None,
                         ApproxFloatNNMethod="pca2nn", **nv):
    """[matches, matchMetric] = matchFeaturesScratch(F1, F2, 'Method','Exhaustive', ...)  (:1-215)

    matches: [K x 2] uint32 (1-based rows of F1 / F2); matchMetric: [K x 1] (SSD, or percent Hamming).
    Method='Approximate' with float descriptors: ApproxFloatNNMethod 'pca2nn' (the parser default, :75), 'subsetpdist2',
    'kdtree' (:128-163), built for Unique=true.  Binary: exhaustive (:611)."""
    ctx = ctx or default_context()
    if str(Method).lower() not in ("exhaustive", "approximate"):
        raise ValueError(f"Unknown Method: {Method}")  # :164-165
    approx = str(Method).lower() == "approximate"
    if not (MaxRatio > 0 and MaxRatio <= 1) or MatchThreshold < 0:
        raise ValueError("invalid MaxRatio / MatchThreshold")  # inputParser validators :60-62
    # normalizeInputs :237-292
    if isinstance(F1, binaryFeatures) and isinstance(F2, binaryFeatures):
        A, B, is_binary = F1.Features, F2.Features, True
    else:
        a, b = np.asarray(F1), np.asarray(F2)

        def isbin(x):
            return x.dtype == np.bool_ or (x.dtype == np.uint8 and bool(np.all((x == 0) | (x == 1))))

        if isbin(a) and isbin(b):
            if a.size == 0 or b.size == 0:
                return np.zeros((0, 2), np.uint32), np.zeros((0,), np.float32)
            if a.shape[1] != b.shape[1]:
                raise ValueError("Descriptor dimensions must match.")
            # unpacked 0/1 bits: packed MSB-first ON THE DEVICE (packBits :617-646), nBits = Dbits
            A, la = _as_matrix(a.astype(np.uint8), np.uint8)
            B, lb = _as_matrix(b.astype(np.uint8), np.uint8)
            if la != lb:
                A, B, la = np.ascontiguousarray(A), np.ascontiguousarray(B), APS_ROW_MAJOR
            N1 = A.shape[0]
            m = np.zeros((max(N1, 1), 2), np.uint32)
            met = np.zeros(max(N1, 1), np.float64)
            K = C.c_int64(0)
            check(lib().aps_match_features_bits(ctx.handle, _ptr(A), N1, _ptr(B), B.shape[0], int(A.shape[1]), la,
                                                float(MatchThreshold), float(MaxRatio), int(bool(Unique)), _ptr(m),
                                                _ptr(met), C.byref(K)))
            return m[:K.value].copy(), met[:K.value].copy()
        else:
            A, B, is_binary = a, b, False
    if approx and not is_binary:
        nn = str(ApproxFloatNNMethod).lower()
        if nn not in ("pca2nn", "kdtree", "subsetpdist2"):
            raise ValueError("Select a approximate method")  # :156-157
        if not Unique:
            raise ApsError(9, "apsmatch:method", "approximate float matching is built for Unique=true only")
        A = np.asarray(A, np.float32)
        B = np.asarray(B, np.float32)
        if A.shape[0] == 0 or B.shape[0] == 0:
            return np.zeros((0, 2), np.uint32), np.zeros((0,), np.float64)
        if A.shape[1] != B.shape[1]:
            raise ValueError("Descriptor dimensions must match for non-binary.")
        plan = PairwisePlan(ctx, [A.shape[0], B.shape[0]], A.shape[1], False)
        try:
            plan.set_method(nn)
            plan.upload([A, B])
            plan.prepare()
            _, rows, met = plan.match(float(MatchThreshold), float(MaxRatio))
        finally:
            plan.close()
        return rows.astype(np.uint32), met
    A, la = _as_matrix(A, np.uint8 if is_binary else np.float32)
    B, lb = _as_matrix(B, np.uint8 if is_binary else np.float32)
    if la != lb:
        A, B, la = np.ascontiguousarray(A), np.ascontiguousarray(B), APS_ROW_MAJOR
    if A.shape[0] and B.shape[0] and A.shape[1] != B.shape[1]:
        raise ValueError("Descriptor dimensions must match for non-binary.")  # :284-286
    N1, N2 = A.shape[0], B.shape[0]
    m = np.zeros((max(N1, 1), 2), np.uint32)
    met = np.zeros(max(N1, 1), np.float64)
    K = C.c_int64(0)
    check(lib().aps_match_features(ctx.handle, _ptr(A), N1, _ptr(B), N2, int(A.shape[1]),
                                   APS_U8 if is_binary else APS_F32, la, float(MatchThreshold), float(MaxRatio),
                                   int(bool(Unique)), _ptr(m), _ptr(met), C.byref(K)))
    return m[:K.value].copy(), met[:K.value].copy()


def flann_knn_win(train, *args, ctx=None):
    """[idx, dist] = flann_knn_win(train, k[,method,trees,checks]) or (train, query, k[,...])

    PP/mex/flann_knn.cpp:118-253.  idx [Fq x k] uint32 1-based, dist [Fq x k] single; float
    descriptors: squared L2 (exact search); uint8: Hamming.  Missing neighbours: 0 / +inf."""
    ctx = ctx or default_context()
    if len(args) < 1:
        raise ApsError(1, "flann_knn:args", "Usage: [idx, dist] = flann_knn(train, k [, method, trees, checks])")
    train = np.asarray(train)
    if train.dtype not in (np.float32, np.uint8):
        raise ApsError(2, "flann_knn:type", "Descriptors must be single (float) or uint8 (binary)")
    args = list(args)
    query = train
    if len(args) >= 2 and isinstance(args[0], np.ndarray) and args[0].dtype == train.dtype and args[0].ndim == 2:
        query = args.pop(0)
    kk = args.pop(0)
    if not np.isscalar(kk):
        raise ApsError(2, "flann_knn:type", "k must be a scalar double")
    k = int(kk)
    method = str(args.pop(0)) if args else "flann"
    trees = int(args.pop(0)) if args else 4
    checks = int(args.pop(0)) if args else 32
    dt = np.float32 if train.dtype == np.float32 else np.uint8
    T, lt = _as_matrix(train, dt)
    Q, lq = (T, lt) if query is train else _as_matrix(query, dt)
    if lt != lq:
        T, Q, lt = np.ascontiguousarray(T), np.ascontiguousarray(Q), APS_ROW_MAJOR
    if T.shape[1] != Q.shape[1]:
        raise ApsError(4, "flann_knn:dim", "query must have same descriptor dimension as train")
    Fq = Q.shape[0]
    order = "C" if lt == APS_ROW_MAJOR else "F"
    idx = np.zeros((Fq, max(k, 1)), np.uint32, order=order)
    dist = np.zeros((Fq, max(k, 1)), np.float32, order=order)
    check(lib().aps_flann_knn(ctx.handle, _ptr(T), T.shape[0], _ptr(Q), Fq, int(T.shape[1]),
                              APS_F32 if dt == np.float32 else APS_U8, lt, k, method.encode(), trees, checks,
                              _ptr(idx), _ptr(dist)))
    return idx, dist


def nearest2HammingExhaustiveMEX(A, B, ctx=None):
    """[idx2, d1, d2] = nearest2HammingExhaustiveMEX(Abytes, Bbytes)  (nearest2HammingExhaustiveMEX.cpp:16-80)"""
    ctx = ctx or default_context()
    A, B = np.asarray(A), np.asarray(B)
    if A.dtype != np.uint8 or B.dtype != np.uint8:
        raise ApsError(2, "hamm2nn:type", "Inputs must be uint8.")
    if A.ndim != 2 or B.ndim != 2:
        raise ApsError(4, "hamm2nn:dim", "2D only.")
    if A.shape[1] != B.shape[1]:
        raise ApsError(4, "hamm2nn:cols", "Byte width mismatch.")
    A, la = _as_matrix(A, np.uint8)
    B, lb = _as_matrix(B, np.uint8)
    if la != lb:
        A, B, la = np.ascontiguousarray(A), np.ascontiguousarray(B), APS_ROW_MAJOR
    N1 = A.shape[0]
    idx2 = np.zeros(N1, np.uint32)
    d1 = np.zeros(N1, np.float32)
    d2 = np.zeros(N1, np.float32)
    check(lib().aps_nearest2_hamming(ctx.handle, _ptr(A), N1, _ptr(B), B.shape[0], int(A.shape[1]), la, _ptr(idx2),
                                     _ptr(d1), _ptr(d2)))
    return idx2, d1, d2


nearest2HammingExhaustiveOMPMEX = nearest2HammingExhaustiveMEX  # same contract (…OMPMEX.cpp:18-83)


def nearest2SSDExhaustive(A, B, ctx=None):
    """[idx1, idx2, d1, d2] = nearest2SSDExhaustive(A, B)  (matchFeaturesScratch.m:322-366)"""
    ctx = ctx or default_context()
    A, la = _as_matrix(A, np.float32)
    B, lb = _as_matrix(B, np.float32)
    if la != lb:
        A, B, la = np.ascontiguousarray(A), np.ascontiguousarray(B), APS_ROW_MAJOR
    N1 = A.shape[0]
    idx2 = np.zeros(N1, np.uint32)
    d1 = np.zeros(N1, np.float32)
    d2 = np.zeros(N1, np.float32)
    check(lib().aps_nearest2_ssd(ctx.handle, _ptr(A), N1, _ptr(B), B.shape[0], int(A.shape[1]), la, _ptr(idx2),
                                 _ptr(d1), _ptr(d2)))
    return np.arange(1, N1 + 1, dtype=np.float64), idx2, d1, d2


def _putative_counts(matchesAll):
    """putativeCount of imageMatching.m:76: rows of every cell of the n x n nested list (or an integer count matrix)"""
    if isinstance(matchesAll, np.ndarray):
        return matchesAll.astype(np.int64)
    n = len(matchesAll)
    return np.array([[np.asarray(matchesAll[i][j]).shape[0] if np.asarray(matchesAll[i][j]).ndim == 2 else 0
                      for j in range(n)] for i in range(n)], np.int64)


def selectImagePartners(matchesAll, m, ctx=None):
    """Top-m candidate selection of imageMatching.m:75-100.

    matchesAll: n x n nested list of [M x 2] arrays (or an [n x n] integer count matrix).
    Returns (candidatePairs [n x n] bool, IuptriIdx: 1-based column-major linear indices)."""
    ctx = ctx or default_context()
    counts = _putative_counts(matchesAll)
    n = counts.shape[0]
    if counts.shape != (n, n):
        raise ValueError("matchesAll must be an n-by-n cell array.")  # imageMatching.m:58-60
    cm = np.ascontiguousarray(counts.T)  # column-major buffer: cm.flat[i + j*n] = counts[i, j]
    cand = np.zeros(n * n, np.uint8)
    pairs = np.zeros(max(n * n, 1), np.int64)
    npairs = C.c_int64(0)
    check(lib().aps_select_partners(ctx.handle, _ptr(cm), n, int(m), _ptr(cand), _ptr(pairs), C.byref(npairs)))
    return cand.reshape(n, n).T.astype(bool), pairs[:npairs.value] + 1


def ransacSampleTable(pt_ptr, n_draws, seed=0, ctx=None):
    """The device generator's table of minimal samples: [n_pairs x n_draws x 4] zero-based indices
    (stand-in for randperm(numPoints, 4), estimateTransformationRANSAC.m:97)."""
    ctx = ctx or default_context()
    pt_ptr = np.ascontiguousarray(pt_ptr, np.int64)
    P = pt_ptr.size - 1
    out = np.zeros((max(P, 0), int(n_draws), 4), np.uint32)
    if P > 0:
        check(lib().aps_ransac_sample_table(ctx.handle, _ptr(pt_ptr), P, int(n_draws), int(seed), _ptr(out)))
    return out


def _ransac_params(input):
    return (float(_field(input, "maxDistance", 2.0)), float(_field(input, "inliersConfidence", 99.9)),
            int(_field(input, "maxIter", 500)))


def imageMatchingBatch(pt_ptr, pts1, pts2, input=None, samples=None, n_draws=None, seed=0, ctx=None):
    """RANSAC homographies for a batch of candidate pairs given as CSR correspondences (aps_image_matching_batch).
    pts1 / pts2: [total x 2] (matchedPoints1 = image jj, matchedPoints2 = image ii).  Returns a dict with
    models / models_inv [P x 3 x 3], inliers bool[total], n_inliers, accepted, draws_used."""
    ctx = ctx or default_context()
    md, conf, mt = _ransac_params(input or {})
    pt_ptr = np.ascontiguousarray(pt_ptr, np.int64)
    P = pt_ptr.size - 1
    p1 = np.ascontiguousarray(pts1, np.float64).reshape(-1, 2)
    p2 = np.ascontiguousarray(pts2, np.float64).reshape(-1, 2)
    total = p1.shape[0]
    if samples is not None:
        samples = np.ascontiguousarray(samples, np.uint32).reshape(P, -1, 4)
        n_draws = samples.shape[1]
    n_draws = int(n_draws or 2 * mt)
    models, minv = np.full((P, 3, 3), np.nan), np.full((P, 3, 3), np.nan)
    inl, ni = np.zeros(max(total, 1), np.uint8), np.zeros(max(P, 1), np.int32)
    acc, du = np.zeros(max(P, 1), np.uint8), np.zeros(max(P, 1), np.int32)
    check(lib().aps_image_matching_batch(ctx.handle, P, _ptr(pt_ptr), _ptr(p1), _ptr(p2), md, conf, mt,
                                         _ptr(samples) if samples is not None else C.c_void_p(0), n_draws, int(seed),
                                         _ptr(models), _ptr(minv), _ptr(inl), _ptr(ni), _ptr(acc), _ptr(du)))
    return dict(models=models, models_inv=minv, inliers=inl[:total].astype(bool), n_inliers=ni[:P],
                accepted=acc[:P].astype(bool), draws_used=du[:P])


def estimateTransformationRANSAC(matchedPoints1, matchedPoints2, transformType="projective", input=None, samples=None,
                                 seed=0, ctx=None):
    """[model, inliers, isFound] = estimateTransformationRANSAC(...) (estimateTransformationRANSAC.m:1-183).
    Only 'projective' (PP/inputs.m:73) is built; model is None where the reference returns []."""
    if str(transformType).lower() != "projective":
        raise ValueError("Unknown transform type" if str(transformType).lower() not in
                         ("affine", "similarity", "rigid", "translation") else
                         f"transform type '{transformType}' is outside the B200 path (projective only)")
    p1 = np.asarray(matchedPoints1, np.float64).reshape(-1, 2)
    p2 = np.asarray(matchedPoints2, np.float64).reshape(-1, 2)
    if p1.shape[0] != p2.shape[0]:
        raise ValueError("matchedPoints1 and matchedPoints2 must have the same number of rows.")  # :51-53
    if samples is not None:
        samples = np.asarray(samples, np.uint32).reshape(1, -1, 4)
    r = imageMatchingBatch([0, p1.shape[0]], p1, p2, input, samples, None, seed, ctx)
    found = bool(np.isfinite(r["models"][0]).all() and r["n_inliers"][0] >= 4)
    return (r["models"][0] if found else None), r["inliers"], found


def imageMatching(input, n, keypoints, matchesAll, imagesProcessed=None, samples=None, seed=0, ctx=None):
    """[allMatches, numMatches, tforms] = imageMatching(input, n, keypoints, matchesAll, imagesProcessed)
    (imageMatching.m:1-156, custom 'ransac' branch): top-m partner selection, RANSAC homography per candidate
    pair on the GPU (matched keypoints gathered on the device from the CSR lists), acceptance ni > 8 + 0.3 nf.
    keypoints: list of [Ni x 2]; matchesAll: n x n nested list of [M x 2] 1-based index pairs.
    Returns nested lists / an [n x n] array like the reference's cells; tforms[i][j] maps image j to image i."""
    ctx = ctx or default_context()
    n = int(n)
    if len(matchesAll) != n or any(len(r) != n for r in matchesAll):
        raise ValueError("matchesAll must be an n-by-n cell array.")  # imageMatching:InvalidMatchesAllSize
    if len(keypoints) != n:
        raise ValueError("keypoints must contain n elements (one per image).")
    if str(_field(input, "imageMatchingMethod", "ransac")).lower() != "ransac" or int(_field(input, "useMATLABImageMatching", 0)):
        raise ValueError("only input.imageMatchingMethod = 'ransac' with useMATLABImageMatching = 0 is built")
    allMatches = [[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)]
    numMatches = np.zeros((n, n))
    tforms = [[None] * n for _ in range(n)]
    _, lin1 = selectImagePartners(matchesAll, int(_field(input, "mBrownLowe", 6)), ctx)
    if lin1.size == 0:
        return allMatches, numMatches, tforms
    lin = np.ascontiguousarray(lin1 - 1, np.int64)
    # CSR of the cell (column-major cell index c = i + j*n), pooled keypoints
    pair_ptr = np.zeros(n * n + 1, np.int64)
    segs = []
    for j in range(n):
        for i in range(n):
            a = np.asarray(matchesAll[i][j])
            cnt = a.shape[0] if (a.ndim == 2 and i < j) else 0
            pair_ptr[i + j * n + 1] = cnt
            if cnt:
                segs.append(np.ascontiguousarray(a, np.float64).astype(np.uint32))
    pair_ptr = np.cumsum(pair_ptr)
    rows = np.ascontiguousarray(np.vstack(segs), np.uint32) if segs else np.zeros((0, 2), np.uint32)
    kps = [np.asarray(k, np.float64).reshape(-1, 2) for k in keypoints]
    img_off = np.concatenate([[0], np.cumsum([k.shape[0] for k in kps])]).astype(np.int64)
    kp = np.ascontiguousarray(np.vstack(kps)) if img_off[-1] else np.zeros((0, 2))
    md, conf, mt = _ransac_params(input)
    P = lin.size
    total = int(sum(pair_ptr[c + 1] - pair_ptr[c] for c in lin))
    if samples is not None:
        samples = np.ascontiguousarray(samples, np.uint32).reshape(P, -1, 4)
    n_draws = samples.shape[1] if samples is not None else 2 * mt
    ptr = np.zeros(P + 1, np.int64)
    models, minv = np.full((P, 3, 3), np.nan), np.full((P, 3, 3), np.nan)
    inl, ni = np.zeros(max(total, 1), np.uint8), np.zeros(P, np.int32)
    acc, du = np.zeros(P, np.uint8), np.zeros(P, np.int32)
    check(lib().aps_image_matching(ctx.handle, n, _ptr(pair_ptr), _ptr(rows), _ptr(kp), _ptr(img_off), _ptr(lin), P, md,
                                   conf, mt, _ptr(samples) if samples is not None else C.c_void_p(0), n_draws, int(seed),
                                   _ptr(ptr), _ptr(models), _ptr(minv), _ptr(inl), _ptr(ni), _ptr(acc), _ptr(du)))
    for p, c in enumerate(lin):
        if not acc[p]:
            continue
        i, j = int(c % n), int(c // n)
        m = np.asarray(matchesAll[i][j], np.float64)
        allMatches[i][j] = m[inl[ptr[p]:ptr[p + 1]].astype(bool)]  # imageMatching.m:148
        numMatches[i, j] = ni[p]
        tforms[i][j], tforms[j][i] = models[p], minv[p]  # :150-151, :165-166
    imageMatching.last = dict(pairs_lin=lin, pt_ptr=ptr, n_inliers=ni, accepted=acc.astype(bool), draws_used=du,
                              models=models, models_inv=minv, inliers=inl[:total].astype(bool))
    return allMatches, numMatches, tforms


def _set_counts(matchesAll):
    c = _putative_counts(matchesAll)
    return c.reshape(0, 0) if c.size == 0 and c.ndim == 1 else c   # a set without images: a 0 x 0 block


def _select_partners_sets(ctx, counts_sets, m):
    """aps_select_partners_sets over [n_b x n_b] count matrices -> (cand blocks, 0-based pairs_lin, set_pair_ptr)"""
    ns = [c.shape[0] for c in counts_sets]
    B, cells = len(ns), sum(n * n for n in ns)
    cm = (np.concatenate([np.ascontiguousarray(c.T).ravel() for c in counts_sets]).astype(np.int64) if cells
          else np.zeros(0, np.int64))  # column-major blocks, set after set
    cand = np.zeros(cells, np.uint8)
    pairs = np.zeros(sum(n * (n - 1) // 2 for n in ns), np.int64)
    spp = np.zeros(B + 1, np.int64)
    simg = (C.c_int * max(B, 1))(*ns)
    check(lib().aps_select_partners_sets(ctx.handle, B, simg, _ptr(cm), int(m), _ptr(cand), _ptr(pairs), _ptr(spp)))
    return cand, pairs[:spp[-1]], spp


def selectImagePartnersSets(matchesAllSets, m, ctx=None):
    """selectImagePartners over B independent image sets in one call (aps_select_partners_sets): element b of the
    returned list is exactly selectImagePartners(matchesAllSets[b], m) -- (candidatePairs, 1-based IuptriIdx)."""
    ctx = ctx or default_context()
    counts = [_set_counts(mb) for mb in matchesAllSets]
    for b, c in enumerate(counts):
        if c.shape != (c.shape[0], c.shape[0]):
            raise ValueError(f"matchesAllSets[{b}] must be an n-by-n cell array.")
    cand, pairs, spp = _select_partners_sets(ctx, counts, m)
    out, c0 = [], 0
    for b, c in enumerate(counts):
        n = c.shape[0]
        out.append((cand[c0:c0 + n * n].reshape(n, n).T.astype(bool), pairs[spp[b]:spp[b + 1]] + 1))
        c0 += n * n
    return out


def imageMatchingSets(input, numImgs, keypointsSets, matchesAllSets, seed=0, samples=None, ctx=None):
    """[allMatchesSets, numMatchesSets, tformsSets] = imageMatchingSets(input, numImgs, keypointsSets, matchesAllSets)

    imageMatching over B independent image sets in one call (aps_select_partners_sets, then aps_image_matching_sets):
    set b is keypointsSets[b] / matchesAllSets[b] with numImgs[b] images.  Returns a list of B tuples, element b exactly
    what imageMatching(input, numImgs[b], keypointsSets[b], matchesAllSets[b], seed=seed) returns.  samples: None (drawn
    on the device, each set as its single-set call draws) or one table per set, each what imageMatching's `samples`
    would be for that set.  Device groups (input.apsGPUs) are not supported here."""
    if _field(input, "apsGPUs", None) is not None:
        raise ValueError("input.apsGPUs is not supported by imageMatchingSets; verify the sets on one GPU")
    kps_sets, m_sets = list(keypointsSets), list(matchesAllSets)
    nums = list(np.atleast_1d(np.asarray(numImgs, dtype=np.float64)).ravel()) if np.size(numImgs) else []
    if len(nums) != len(kps_sets) or len(nums) != len(m_sets):
        raise ValueError("numImgs must give one image count per keypoint set and per match set")
    for v in nums:
        if not (np.isfinite(v) and v >= 0 and v == np.round(v)):
            raise ValueError("every numImgs entry must be a non-negative integer")
    if str(_field(input, "imageMatchingMethod", "ransac")).lower() != "ransac" or int(_field(input, "useMATLABImageMatching", 0)):
        raise ValueError("only input.imageMatchingMethod = 'ransac' with useMATLABImageMatching = 0 is built")
    if str(_field(input, "transformationType", "projective")).lower() != "projective":
        raise ValueError("only input.transformationType = 'projective' is built")
    ns = [int(v) for v in nums]
    for b, (n, kps, mall) in enumerate(zip(ns, kps_sets, m_sets)):
        if len(mall) != n or any(len(r) != n for r in mall):
            raise ValueError(f"matchesAllSets[{b}] must be an n-by-n cell array.")  # imageMatching:InvalidMatchesAllSize
        if len(kps) != n:
            raise ValueError(f"keypointsSets[{b}] must contain n elements (one per image).")
    ctx = ctx or default_context()
    B = len(ns)
    _, lin, spp = _select_partners_sets(ctx, [_set_counts(mall) for mall in m_sets], int(_field(input, "mBrownLowe", 6)))
    result = [([[np.zeros((0, 0)) for _ in range(n)] for _ in range(n)], np.zeros((n, n)), [[None] * n for _ in range(n)])
              for n in ns]
    imageMatchingSets.last = [dict(pairs_lin=np.zeros(0, np.int64), pt_ptr=np.zeros(1, np.int64)) for _ in ns]
    P = int(spp[-1])
    if P == 0:
        return result
    # per set: CSR of the cell (column-major cell index c = i + j*n, strict upper triangle), as imageMatching builds it
    pps, rows = [], []
    for n, mall in zip(ns, m_sets):
        pp, segs = np.zeros(n * n + 1, np.int64), []
        for j in range(n):
            for i in range(j):
                a = np.asarray(mall[i][j])
                if a.ndim == 2 and a.shape[0]:
                    pp[i + j * n + 1] = a.shape[0]
                    segs.append(np.ascontiguousarray(a, np.float64).astype(np.uint32))
        pps.append(np.cumsum(pp))
        rows.append(np.ascontiguousarray(np.vstack(segs), np.uint32) if segs else np.zeros((0, 2), np.uint32))
    kps = [np.asarray(k, np.float64).reshape(-1, 2) for ks in kps_sets for k in ks]
    img_off = np.concatenate([[0], np.cumsum([k.shape[0] for k in kps], dtype=np.int64)]).astype(np.int64)
    kp = np.ascontiguousarray(np.vstack(kps)) if img_off[-1] else np.zeros((0, 2))
    md, conf, mt = _ransac_params(input)
    n_draws = 2 * mt
    if samples is not None:
        tabs = [np.ascontiguousarray(t, np.uint32) for t in samples]
        if len(tabs) != B:
            raise ValueError("samples must hold one table per set")
        n_draws = next((t.size // (4 * (spp[b + 1] - spp[b])) for b, t in enumerate(tabs) if spp[b + 1] > spp[b]), 0)
        samples = np.ascontiguousarray(np.concatenate([t.reshape(spp[b + 1] - spp[b], n_draws, 4)
                                                       for b, t in enumerate(tabs)]))
    ptr = np.zeros(P + 1, np.int64)
    total = 0
    for b in range(B):
        total += int(sum(pps[b][c + 1] - pps[b][c] for c in lin[spp[b]:spp[b + 1]]))
    models, minv = np.full((P, 3, 3), np.nan), np.full((P, 3, 3), np.nan)
    inl, ni = np.zeros(total, np.uint8), np.zeros(P, np.int32)
    acc, du = np.zeros(P, np.uint8), np.zeros(P, np.int32)
    simg = (C.c_int * B)(*ns)
    pp_arr = (C.c_void_p * B)(*[p.ctypes.data for p in pps])
    rows_arr = (C.c_void_p * B)(*[r.ctypes.data if r.size else None for r in rows])
    check(lib().aps_image_matching_sets(ctx.handle, B, simg, pp_arr, rows_arr, _ptr(kp), _ptr(img_off), _ptr(spp),
                                        _ptr(lin), md, conf, mt, _ptr(samples) if samples is not None else C.c_void_p(0),
                                        int(n_draws), int(seed), _ptr(ptr), _ptr(models), _ptr(minv), _ptr(inl), _ptr(ni),
                                        _ptr(acc), _ptr(du)))
    for b, (n, mall) in enumerate(zip(ns, m_sets)):
        p0, p1 = int(spp[b]), int(spp[b + 1])
        allMatches, numMatches, tforms = result[b]
        for p in range(p0, p1):
            if not acc[p]:
                continue
            c = lin[p]
            i, j = int(c % n), int(c // n)
            mij = np.asarray(mall[i][j], np.float64)
            allMatches[i][j] = mij[inl[ptr[p]:ptr[p + 1]].astype(bool)]  # imageMatching.m:148
            numMatches[i, j] = ni[p]
            tforms[i][j], tforms[j][i] = models[p], minv[p]  # :150-151, :165-166
        t0, t1 = ptr[p0], ptr[p1]
        imageMatchingSets.last[b] = dict(pairs_lin=lin[p0:p1], pt_ptr=ptr[p0:p1 + 1] - t0, n_inliers=ni[p0:p1],
                                         accepted=acc[p0:p1].astype(bool), draws_used=du[p0:p1], models=models[p0:p1],
                                         models_inv=minv[p0:p1], inliers=inl[t0:t1].astype(bool))
    return result


RECORD_PAD = 16384  # APS_RECORD_PAD of include/apsmatch.h: rows the record buffer holds beyond F


def _csr_from_matchlist(h, n):
    L = lib()
    total = L.aps_matchlist_total(h)
    pp = np.ctypeslib.as_array(L.aps_matchlist_pair_ptr(h), shape=(n * n + 1,)).copy()
    rows = (np.ctypeslib.as_array(L.aps_matchlist_rows(h), shape=(total, 2)).copy() if total
            else np.zeros((0, 2), np.uint32))
    mp = L.aps_matchlist_metric(h)
    met = np.ctypeslib.as_array(mp, shape=(total,)).copy() if (total and mp) else np.zeros(0)
    return pp, rows, met


class PairwisePlan:
    """Staged pairwise pipeline (aps_pplan_*): descriptors resident on the device, K1 once, then this rank's share of
    the image-pair list -- what PP/featureMatching/featureMatchingPairwise.m:48-59 does with a parfor over the pairs
    after broadcasting the descriptor cell to the workers."""

    def __init__(self, ctx, counts, D, is_binary):
        self.ctx, self.n, self.D = ctx, len(counts), int(D)
        h = C.c_void_p()
        cnt = (C.c_int64 * max(self.n, 1))(*[int(c) for c in counts])
        check(lib().aps_pplan_create(ctx.handle, cnt, self.n, self.D, APS_U8 if is_binary else APS_F32, C.byref(h)))
        self._h = h
        self.F = int(lib().aps_pplan_total(h))

    def upload(self, mats):
        ptrs, _, layout, keep = _desc_args(list(mats), [0 if m is None else m.shape[0] for m in mats])
        check(lib().aps_pplan_upload(self._h, ptrs, layout))
        self._keep = keep

    def desc_device(self):
        return lib().aps_pplan_desc_device(self._h)

    def set_method(self, method, subset=12000, seed=0):
        """'exhaustive' | 'subsetpdist2' | 'kdtree' (aps_method, include/apsmatch.h; matchFeaturesScratch.m:116-163).
        Call before prepare()."""
        self.subset = int(subset)
        check(lib().aps_pplan_set_method(self._h, APS_METHOD[str(method).lower()], int(subset), int(seed)))

    def subset_table(self, image):
        """candB of a train image above the subset size: `subset` distinct 0-based rows (after prepare())."""
        out = np.zeros(self.subset, np.int32)
        check(lib().aps_pplan_subset_table(self._h, int(image), _ptr(out)))
        return out

    def prepare(self):
        """K1 of the pairwise path: magnitude test per image (matchFeaturesScratch.m:105-110), norms, tensor operands."""
        check(lib().aps_pplan_prepare(self._h))

    def match(self, match_threshold, max_ratio, first=0, stride=1):
        """This rank's share of the pair list -> CSR (pair_ptr [n*n+1], rows [M x 2] uint32, metric [M])."""
        h = C.c_void_p()
        check(lib().aps_pplan_match(self._h, float(match_threshold), float(max_ratio), int(first), int(stride), C.byref(h)))
        try:
            return _csr_from_matchlist(h, self.n)
        finally:
            lib().aps_matchlist_free(h)

    def close(self):
        if getattr(self, "_h", None):
            lib().aps_pplan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GlobalPlan:
    """Staged global pipeline (aps_gplan_*): the building block bench.py and the multi-GPU host use.

    The stages of PP/featureMatching/featureMatchingGlobal.m as separate calls: pooling + normalisation :70-97
    (upload / prepare), global kNN :106-120 (knn), per-feature filter loop :123-161 (filter, then compact once the
    ranks have exchanged their record slices)."""

    def __init__(self, ctx, counts, D, is_binary, k):
        self.ctx, self.n, self.D, self.k = ctx, len(counts), int(D), int(k)
        self.counts = np.asarray(counts, np.int64)
        self.is_binary = bool(is_binary)
        h = C.c_void_p()
        cnt = (C.c_int64 * max(self.n, 1))(*[int(c) for c in counts])
        check(lib().aps_gplan_create(ctx.handle, cnt, self.n, self.D, APS_U8 if is_binary else APS_F32, self.k,
                                     C.byref(h)))
        self._h = h
        self.F = int(lib().aps_gplan_total(h))

    def upload(self, mats):
        """H2D of the per-image descriptor matrices into the pooled [F x D] matrix (vertcat, featureMatchingGlobal.m:70-77)."""
        ptrs, _, layout, keep = _desc_args(list(mats), [0 if m is None else m.shape[0] for m in mats])
        check(lib().aps_gplan_upload(self._h, ptrs, layout))
        self._keep = keep

    def upload_pointers(self, ptr_list, layout=APS_ROW_MAJOR):
        """Same from raw host pointers (pinned staging buffers of aps_host_alloc), one per image."""
        ptrs = (C.c_void_p * max(self.n, 1))(*ptr_list)
        check(lib().aps_gplan_upload(self._h, ptrs, layout))

    def desc_device(self):
        """Device pointer of the pooled descriptors (for the NCCL all-gather of row blocks, multigpu.gather_descriptors)."""
        return lib().aps_gplan_desc_device(self._h)

    def records_device(self):
        """Device pointer of the per-query records: [F + RECORD_PAD] x (int32 target image, uint32 partner) (the accept / match of :140-152)."""
        return lib().aps_gplan_records_device(self._h)

    def knn_device(self):
        """Device pointers (idx, dist) of the [F x k] kNN tables (nnIdxAll / nnDistAll, :106-120)."""
        return lib().aps_gplan_knn_idx_device(self._h), lib().aps_gplan_knn_dist_device(self._h)

    def prepare(self):
        """K1: single + L2 normalisation with eps inside the sqrt (:80-84), tensor operands, train view."""
        check(lib().aps_gplan_prepare(self._h))

    def knn(self, q0=0, q1=None):
        """K2/K3 (or K4 for binary): exact k nearest neighbours of query rows [q0, q1) against all F rows (:106-120)."""
        check(lib().aps_gplan_knn(self._h, int(q0), int(self.F if q1 is None else q1)))

    def filter(self, ratio, q0=0, q1=None):
        """K5a: self / same-image removal and Lowe ratio test of rows [q0, q1) (:123-147) -> records."""
        check(lib().aps_gplan_filter(self._h, int(q0), int(self.F if q1 is None else q1), float(ratio)))

    def filter_mutual(self):
        """Opt-in cross-check of the complete record set (not reference behaviour, see include/apsmatch.h)."""
        check(lib().aps_gplan_filter_mutual(self._h))

    def compact(self):
        """K5b: scatter of all F records into the n x n cell in the reference's loop order (:149-159), CSR form."""
        check(lib().aps_gplan_compact(self._h))

    def download_knn(self, q0=0, q1=None):
        """D2H of the kNN tables of rows [q0, q1): (idx uint32 1-based, dist float32), as flann_knn_win returns them."""
        q1 = self.F if q1 is None else q1
        idx = np.zeros((max(q1 - q0, 0), self.k), np.uint32)
        dist = np.zeros((max(q1 - q0, 0), self.k), np.float32)
        check(lib().aps_gplan_download_knn(self._h, int(q0), int(q1), _ptr(idx), _ptr(dist)))
        return idx, dist

    def download(self):
        """D2H of the CSR match lists (pair_ptr, rows) -- the `matches` cell of featureMatchingGlobal.m:155-159."""
        h = C.c_void_p()
        check(lib().aps_gplan_download(self._h, C.byref(h)))
        try:
            return _cells_from_matchlist(h, self.n)
        finally:
            lib().aps_matchlist_free(h)

    def close(self):
        if getattr(self, "_h", None):
            lib().aps_gplan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
