"""featureMatchingGlobal over many image sets in one call (aps_feature_matching_global_sets) without a GPU: the arguments
are checked before any device is touched and keep the single-set call's MATLAB ids, a well-formed call fails with
apsmatch:nogpu (no CPU fallback), the host mirror rejects input.apsGPUs, and the MEX verb 'globalsets' checks its
arguments under the mex shim."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _library(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    return aps._lib.lib()


def _no_gpu(aps):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by tests/test_gpu_global_sets.py")
    return _library(aps)


def _call(L, nsets, set_images, counts, D=8, dtype=0, k=4, out=True):
    si = (C.c_int * max(len(set_images), 1))(*set_images)
    cnt = (C.c_int64 * max(len(counts), 1))(*counts)
    ptrs = (C.c_void_p * max(len(counts), 1))()
    outs = (C.c_void_p * max(nsets, 1))()
    rc = L.aps_feature_matching_global_sets(None, nsets, si, ptrs, cnt, D, dtype, 1, k, 0.6, 0, 0,
                                            outs if out else None)
    return rc, L.aps_error_id().decode()


@pytest.mark.parametrize("case, code, ident", [
    (dict(nsets=-1, set_images=[], counts=[]), 1, ""),                           # APS_ERR_ARGS
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], out=False), 1, ""),
    (dict(nsets=2, set_images=[1, -1], counts=[4]), 1, ""),
    (dict(nsets=2, set_images=[2, 1], counts=[4, -3, 4]), 1, ""),
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], k=0), 3, "flann_knn:k"),    # APS_ERR_K
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], k=33), 3, "flann_knn:k"),
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], dtype=5), 2, "flann_knn:type"),  # APS_ERR_TYPE
    (dict(nsets=2, set_images=[1, 1], counts=[4, 4], D=0), 4, "flann_knn:dim"),  # APS_ERR_DIM
])
def test_argument_errors_and_their_ids(aps, case, code, ident):
    L = _library(aps)
    rc, got = _call(L, **case)
    assert (rc, got) == (code, ident)


def test_well_formed_call_without_gpu_is_nogpu(aps):
    L = _no_gpu(aps)
    assert _call(L, 2, [1, 1], [0, 0]) == (6, "apsmatch:nogpu")                  # APS_ERR_NOGPU, empty sets included
    import numpy as np

    with pytest.raises(aps.ApsError) as e:
        aps.featureMatchingGlobalSets({"k": 4, "Ratiothreshold": 0.6}, [[np.ones((4, 8), np.float32)]] * 2, [1, 1])
    assert e.value.identifier == "apsmatch:nogpu"


def test_all_empty_sets_need_no_device(aps):
    import numpy as np

    got = aps.featureMatchingGlobalSets({"k": 4, "Ratiothreshold": 0.6}, [[np.zeros((0, 8), np.float32)] * 2, []],
                                        [2, 3])
    assert [len(g) for g in got] == [2, 3]
    assert all(np.asarray(c).size == 0 for g in got for row in g for c in row)


def test_host_rejects_apsGPUs_and_malformed_counts(aps):
    import numpy as np

    sets = [[np.ones((4, 8), np.float32)]] * 2
    with pytest.raises(ValueError, match="apsGPUs"):
        aps.featureMatchingGlobalSets({"k": 4, "Ratiothreshold": 0.6, "apsGPUs": [1]}, sets, [1, 1])
    for bad in ([1], [1, 0], [1, 1.5], [1, float("nan")]):
        with pytest.raises(ValueError, match="numImgs"):
            aps.featureMatchingGlobalSets({"k": 4, "Ratiothreshold": 0.6}, sets, bad)
    with pytest.raises(aps.ApsError) as e:   # one descriptor kind and width for every set
        aps.featureMatchingGlobalSets({"k": 4, "Ratiothreshold": 0.6}, [sets[0], [np.ones((4, 16), np.float32)]], [1, 1])
    assert e.value.identifier == "flann_knn:dim"
    with pytest.raises(aps.ApsError) as e:
        aps.featureMatchingGlobalSets({"k": 4, "Ratiothreshold": 0.6},
                                      [sets[0], [aps.binaryFeatures(np.ones((4, 8), np.uint8))]], [1, 1])
    assert e.value.identifier == "flann_knn:type"


def test_symbol_is_declared_and_bound(aps):
    L = _library(aps)
    assert "aps_feature_matching_global_sets" in L._aps_symbols
    assert "aps_feature_matching_global_sets" in open(os.path.join(ROOT, "include", "apsmatch.h")).read()
    assert "featureMatchingGlobalSets" in dir(aps)


def test_gateway_globalsets_argument_checks(aps):
    import torch

    _library(aps)
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    args = ["sets"] + ([] if torch.cuda.is_available() else ["nogpu"])
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_batched")] + args, capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
