"""Device input (the *_dev entries of include/apsmatch.h) without a GPU: every entry is declared, exported and bound; the
host entry's statuses come first, in its order, then APS_ERR_TYPE for a bad keypoint type, APS_ERR_ARGS for a NULL
device pointer, then the context (apsmatch:nogpu: there is no CPU path); the Python forms refuse host tensors before
touching a device; the keypoint-widening kernel compiles for sm_100a without local memory."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "automaticpanoramicimagestitching-autopanostitch-matlab_b200", "csrc")
ENTRIES = ("aps_feature_matching_global_sets_dev", "aps_feature_matching_pairwise_sets_dev",
           "aps_global_image_matching_sets_dev", "aps_pairwise_image_matching_sets_dev")
PYTHON = ("featureMatchingGlobalSetsDevice", "featureMatchingPairwiseSetsDevice", "featureMatchingPairwiseDevice",
          "globalImageMatchingSetsDevice", "globalImageMatchingDevice", "pairwiseImageMatchingSetsDevice",
          "pairwiseImageMatchingDevice", "featureMatchingGlobalDevice")
FAKE_DEV = 0x7F0000000000   # never dereferenced: every call below fails before any device work


def _library(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    return aps._lib.lib()


def _call(L, entry, nsets=2, set_images=(2, 1), D=4, dtype=0, k=4, method=0, subset=12000, max_trials=500,
          confidence=99.9, pooled=FAKE_DEV, keypoints=FAKE_DEV, kp_dtype=0, out=True):
    nimg = max(sum(max(s, 0) for s in set_images), 1)
    cnt = (C.c_int64 * nimg)(*([3] * nimg))
    si = (C.c_int * max(len(set_images), 1))(*set_images)
    d, kp = C.c_void_p(pooled), C.c_void_p(keypoints)
    outs = (C.c_void_p * max(nsets, 1))() if out else None
    h = C.c_void_p()
    ho = C.byref(h) if out else None
    ransac = (6, 5.5, confidence, max_trials, 0, 0, None, ho)
    if entry == "aps_feature_matching_global_sets_dev":
        rc = L.aps_feature_matching_global_sets_dev(None, nsets, si, d, cnt, D, dtype, k, 0.8, 0, 0, None, outs)
    elif entry == "aps_feature_matching_pairwise_sets_dev":
        rc = L.aps_feature_matching_pairwise_sets_dev(None, nsets, si, d, cnt, D, dtype, 1.5, 0.8, method, subset, 0,
                                                      None, outs)
    elif entry == "aps_global_image_matching_sets_dev":
        rc = L.aps_global_image_matching_sets_dev(None, nsets, si, d, cnt, D, dtype, k, 0.8, 0, 0, kp, kp_dtype, *ransac)
    else:
        rc = L.aps_pairwise_image_matching_sets_dev(None, nsets, si, d, cnt, D, dtype, 1.5, 0.8, method, subset, 0, kp,
                                                    kp_dtype, *ransac)
    return rc, L.aps_error_id().decode()


def test_entries_are_declared_bound_and_exported(aps):
    L = _library(aps)
    hdr = open(os.path.join(ROOT, "include", "apsmatch.h")).read()
    for sym in ENTRIES + ("aps_feature_matching_global_dev",):
        assert sym in L._aps_symbols and sym in hdr, sym
    for name in PYTHON:
        assert callable(getattr(aps, name)), name


COMMON = [
    (dict(nsets=-1, set_images=()), (1, "")),
    (dict(set_images=(2, -1)), (1, "")),
    (dict(dtype=7), None),                         # the host entry's type status
    (dict(D=0), None),                             # ... and its dimension status
    (dict(pooled=0), (1, "")),                     # NULL device pointer with rows
    (dict(), (6, "apsmatch:nogpu")),               # well formed: the context (NULL here) -- no CPU path
    (dict(nsets=0, set_images=()), (6, "apsmatch:nogpu")),
    (dict(set_images=(2, 1), pooled=0, D=0), None),          # the host statuses come before the NULL pointer
]


def _want(entry, case, want):
    if want is not None:
        return want
    glob = "global" in entry
    if "dtype" in case:
        return (2, "flann_knn:type") if glob else (2, "")
    return (4, "flann_knn:dim") if glob else (4, "")


@pytest.mark.parametrize("entry", ENTRIES)
@pytest.mark.parametrize("case, want", COMMON)
def test_statuses_in_the_host_entry_order(aps, entry, case, want):
    assert _call(_library(aps), entry, **case) == _want(entry, case, want)


@pytest.mark.parametrize("entry, case, want", [
    ("aps_feature_matching_global_sets_dev", dict(k=0, pooled=0), (3, "flann_knn:k")),
    ("aps_feature_matching_global_sets_dev", dict(k=33), (3, "flann_knn:k")),
    ("aps_feature_matching_global_sets_dev", dict(out=False), (1, "")),
    ("aps_feature_matching_pairwise_sets_dev", dict(method=9, pooled=0), (9, "")),
    ("aps_feature_matching_pairwise_sets_dev", dict(subset=0), (1, "")),
    ("aps_global_image_matching_sets_dev", dict(k=0), (3, "flann_knn:k")),
    ("aps_global_image_matching_sets_dev", dict(max_trials=0, kp_dtype=7, pooled=0), (1, "")),
    ("aps_global_image_matching_sets_dev", dict(confidence=100.0), (1, "")),
    ("aps_global_image_matching_sets_dev", dict(keypoints=0, kp_dtype=7, pooled=0), (1, "")),
    ("aps_global_image_matching_sets_dev", dict(kp_dtype=7, pooled=0), (2, "")),
    ("aps_global_image_matching_sets_dev", dict(kp_dtype=1), (6, "apsmatch:nogpu")),
    ("aps_global_image_matching_sets_dev", dict(out=False, pooled=0), (1, "")),
    ("aps_pairwise_image_matching_sets_dev", dict(method=9, max_trials=0), (9, "")),
    ("aps_pairwise_image_matching_sets_dev", dict(max_trials=0, kp_dtype=7), (1, "")),
    ("aps_pairwise_image_matching_sets_dev", dict(keypoints=0, kp_dtype=7), (1, "")),
    ("aps_pairwise_image_matching_sets_dev", dict(kp_dtype=7, pooled=0), (2, "")),
    ("aps_pairwise_image_matching_sets_dev", dict(kp_dtype=1), (6, "apsmatch:nogpu")),
])
def test_entry_specific_statuses(aps, entry, case, want):
    assert _call(_library(aps), entry, **case) == want


def test_existing_device_entry_checks_the_context_first(aps):
    L = _library(aps)
    cnt = (C.c_int64 * 1)(3)
    h = C.c_void_p()
    assert L.aps_feature_matching_global_dev(None, None, cnt, 1, 4, 0, 0, 0.8, 0, C.byref(h)) == 6
    assert L.aps_error_id().decode() == "apsmatch:nogpu"


def test_python_forms_refuse_host_tensors(aps):
    torch = pytest.importorskip("torch")
    d = [torch.ones((3, 4)), torch.ones((3, 4))]
    kp = [torch.zeros((3, 2)), torch.zeros((3, 2))]
    inp = {"k": 4, "Ratiothreshold": 0.8, "Matchingthreshold": 1.5, "useMATLABFeatureMatch": 0}
    with pytest.raises(TypeError):
        aps.featureMatchingGlobalSetsDevice(inp, [d], [2])
    with pytest.raises(TypeError):
        aps.featureMatchingPairwiseDevice(inp, d, 2)
    with pytest.raises(TypeError):
        aps.globalImageMatchingDevice(inp, d, 2, kp)
    with pytest.raises(TypeError):
        aps.pairwiseImageMatchingSetsDevice(inp, [d], [2], [kp])
    with pytest.raises(TypeError):     # an array passed by mistake: refused before anything is read from it
        aps.featureMatchingGlobalSetsDevice(inp, [[np.ones((3, 4), np.float32)] * 2], [2])
    with pytest.raises(ValueError, match="numImgs"):
        aps.featureMatchingGlobalSetsDevice(inp, [d], [0])
    with pytest.raises(ValueError):
        aps.globalImageMatchingSetsDevice(dict(inp, apsGPUs=[1]), [d], [2], [kp])


def test_all_empty_sets_need_no_device(aps):
    # featureMatchingGlobal / featureMatchingPairwise on sets without descriptors: cell(numImg), nothing on the device
    got = aps.featureMatchingGlobalSetsDevice({"k": 4, "Ratiothreshold": 0.8}, [[None, None], [None]], [2, 1])
    assert [len(g) for g in got] == [2, 1] and all(c.size == 0 for g in got for row in g for c in row)
    m, metrics = aps.featureMatchingPairwiseDevice({"Matchingthreshold": 1.5, "Ratiothreshold": 0.8,
                                                    "useMATLABFeatureMatch": 0}, [None, None], 2, return_metric=True)
    assert len(m) == 2 and metrics[0][1] is None


def test_widening_kernel_compiles_without_local_memory(tmp_path):
    nvcc = shutil.which("nvcc")
    if nvcc is None:
        pytest.skip("nvcc is not available")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xptxas", "-v", "-c",
                        "-o", str(tmp_path / "g.o"), os.path.join(CSRC, "aps_global_image_matching.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-4000:]
    found, name = {}, None
    for line in r.stderr.splitlines():
        m = re.search(r"Compiling entry function '(\S+)'", line)
        if m:
            name = m.group(1)
            continue
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)
        if m and name:
            found[name] = tuple(int(v) for v in m.groups())
    hits = [v for n, v in found.items() if "k_widen_keypoints" in n]
    assert hits, sorted(found)
    assert all(v == (0, 0, 0) for v in hits), hits
