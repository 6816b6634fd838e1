"""featureMatchingPairwise over many image sets in one call (aps_feature_matching_pairwise_sets) without a GPU: the
arguments are checked before any device is touched and keep the single-set call's statuses, the pooled row limit
(subset views included) is named, a well-formed call fails with apsmatch:nogpu (no CPU fallback), the host mirror
rejects input.apsGPUs and malformed numImgs, and the MEX verb 'pairwisesets' checks its arguments under the mex shim."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INP = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.7, "useMATLABFeatureMatch": 0}


def _library(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    return aps._lib.lib()


def _no_gpu(aps):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by tests/test_gpu_pairwise_sets.py")
    return _library(aps)


def _call(L, nsets, set_images, counts, D=8, dtype=0, method=0, subset=12000, out=True):
    si = (C.c_int * max(len(set_images), 1))(*set_images)
    cnt = (C.c_int64 * max(len(counts), 1))(*counts)
    ptrs = (C.c_void_p * max(len(counts), 1))()
    outs = (C.c_void_p * max(nsets, 1))()
    rc = L.aps_feature_matching_pairwise_sets(None, nsets, si, ptrs, cnt, D, dtype, 1, 1.5, 0.7, method, subset, 0,
                                              outs if out else None)
    return rc, L.aps_last_error().decode()


@pytest.mark.parametrize("case, code", [
    (dict(nsets=-1, set_images=[], counts=[]), 1),                                # APS_ERR_ARGS
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], out=False), 1),
    (dict(nsets=2, set_images=[1, -1], counts=[4]), 1),
    (dict(nsets=2, set_images=[2, 1], counts=[4, -3, 4]), 1),
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], subset=0), 1),
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], dtype=5), 2),                # APS_ERR_TYPE
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], D=0), 4),                    # APS_ERR_DIM
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], method=4), 9),               # APS_ERR_METHOD
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], method=-1), 9),
])
def test_argument_errors_and_their_statuses(aps, case, code):
    L = _library(aps)
    rc, _ = _call(L, **case)
    assert rc == code
    assert L.aps_error_id().decode() == ""   # the single-set pairwise call's errors carry no MATLAB id


def test_pooled_row_limit_counts_the_subset_views(aps):
    """2^31 - 512 rows for the pooled plan: 2 x 2^30 rows pass the check only without 'subsetpdist2' views"""
    L = _library(aps)
    half = (1 << 30) - 300
    rc, msg = _call(L, 2, [1, 1], [half, half], method=1, subset=1000)
    assert rc == 1 and "2^31 - 512" in msg
    rc, msg = _call(L, 2, [1, 1], [1 << 30, 1 << 30])
    assert rc == 1 and "2^31 - 512" in msg


def test_well_formed_call_without_gpu_is_nogpu(aps):
    L = _no_gpu(aps)
    rc, _ = _call(L, 2, [1, 1], [0, 0])
    assert (rc, L.aps_error_id().decode()) == (6, "apsmatch:nogpu")   # APS_ERR_NOGPU, empty sets included
    with pytest.raises(aps.ApsError) as e:
        aps.featureMatchingPairwiseSets(INP, [[np.ones((4, 8), np.float32)] * 2] * 2, [2, 2])
    assert e.value.identifier == "apsmatch:nogpu"


def test_all_empty_sets_need_no_device(aps):
    got = aps.featureMatchingPairwiseSets(INP, [[np.zeros((0, 8), np.float32)] * 2, []], [2, 3])
    assert [len(g) for g in got] == [2, 3]
    assert all(np.asarray(c).size == 0 for g in got for row in g for c in row)
    got, met = aps.featureMatchingPairwiseSets(INP, [[], []], [2, 1], return_metric=True)[0]
    assert len(got) == 2 and met[0][1] is None


def test_host_rejects_apsGPUs_and_malformed_counts(aps):
    sets = [[np.ones((4, 8), np.float32)] * 2] * 2
    with pytest.raises(ValueError, match="apsGPUs"):
        aps.featureMatchingPairwiseSets(dict(INP, apsGPUs=[1]), sets, [2, 2])
    for bad in ([2], [2, 0], [2, 1.5], [2, float("nan")]):
        with pytest.raises(ValueError, match="numImgs"):
            aps.featureMatchingPairwiseSets(INP, sets, bad)
    with pytest.raises(ValueError):
        aps.featureMatchingPairwiseSets(dict(INP, Matchingmethod="Approximate", ApproxFloatNNMethod="lsh"), sets, [2, 2])
    with pytest.raises(aps.ApsError) as e:   # one descriptor kind and width for every set
        aps.featureMatchingPairwiseSets(INP, [sets[0], [np.ones((4, 16), np.float32)]], [2, 1])
    assert e.value.identifier == "flann_knn:dim"
    with pytest.raises(aps.ApsError) as e:
        aps.featureMatchingPairwiseSets(INP, [sets[0], [aps.binaryFeatures(np.ones((4, 8), np.uint8))]], [2, 1])
    assert e.value.identifier == "flann_knn:type"


def test_semantics_warning_as_the_single_set_call(aps):
    with pytest.warns(aps.ApsSemanticsWarning):
        aps.featureMatchingPairwiseSets(dict(INP, useMATLABFeatureMatch=1), [[], []], [2, 2])


def test_symbol_is_declared_and_bound(aps):
    L = _library(aps)
    assert "aps_feature_matching_pairwise_sets" in L._aps_symbols
    assert "aps_feature_matching_pairwise_sets" in open(os.path.join(ROOT, "include", "apsmatch.h")).read()
    assert "featureMatchingPairwiseSets" in dir(aps)


def test_gateway_pairwisesets_argument_checks(aps):
    import torch

    _library(aps)
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    args = ["sets"] + ([] if torch.cuda.is_available() else ["nogpu"])
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_batched")] + args, capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
