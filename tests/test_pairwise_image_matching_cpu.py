"""featureMatchingPairwise + imageMatching in one call (aps_pairwise_image_matching[_sets]) without a GPU: argument
errors are raised before any device is touched and carry the statuses of aps_feature_matching_pairwise_sets, a
well-formed call fails with apsmatch:nogpu (no CPU fallback), the host mirror rejects 'mlesac', non-projective models,
input.apsGPUs and unknown methods, the gateway aps_pairwiseImageMatching_mex checks its arguments under the mex shim,
and the new kernels compile for sm_100a without local-memory spills."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "automaticpanoramicimagestitching-autopanostitch-matlab_b200", "csrc")
INP = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.8, "useMATLABFeatureMatch": 0,
       "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}


def _library(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    return aps._lib.lib()


def _call(L, nsets=2, set_images=(2, 1), D=4, dtype=0, method=0, subset=12000, rows=3, max_trials=500,
          confidence=99.9, keypoints=True, out=True, one=False):
    counts = [rows] * max(sum(max(s, 0) for s in set_images), 1)
    desc = np.zeros((3, max(D, 1)), np.float32)
    ptrs = (C.c_void_p * len(counts))(*([desc.ctypes.data] * len(counts)))
    cnt = (C.c_int64 * len(counts))(*counts)
    kp = np.zeros((3, 2))   # read only after the context
    h = C.c_void_p()
    tail = (1.5, 0.8, method, subset, 0, C.c_void_p(kp.ctypes.data) if keypoints else None, 6, 5.5, confidence,
            max_trials, 0, 0, C.byref(h) if out else None)
    if one:
        rc = L.aps_pairwise_image_matching(None, ptrs, cnt, set_images[0], D, dtype, 1, *tail)
    else:
        si = (C.c_int * max(len(set_images), 1))(*set_images)
        rc = L.aps_pairwise_image_matching_sets(None, nsets, si, ptrs, cnt, D, dtype, 1, *tail)
    return rc, L.aps_error_id().decode()


def test_symbols_are_declared_and_bound(aps):
    L = _library(aps)
    hdr = open(os.path.join(ROOT, "include", "apsmatch.h")).read()
    for sym in ("aps_pairwise_image_matching_sets", "aps_pairwise_image_matching"):
        assert sym in L._aps_symbols and sym in hdr
    assert L.aps_abi_version() == 1
    assert "pairwiseImageMatchingSets" in dir(aps) and "pairwiseImageMatching" in dir(aps)


@pytest.mark.parametrize("case, want", [
    (dict(nsets=-1, set_images=()), (1, "")),
    (dict(set_images=(2, -1)), (1, "")),
    (dict(rows=-1), (1, "")),
    (dict(dtype=7), (2, "")),
    (dict(method=4), (9, "")),
    (dict(method=-1), (9, "")),
    (dict(subset=0), (1, "")),
    (dict(rows=(1 << 30)), (1, "")),                  # pooled rows past 2^31 - 512
    (dict(nsets=1, set_images=(2,), method=1, subset=400, rows=(1 << 30) - 600), (1, "")),  # subset views count
    (dict(D=0), (4, "")),
    (dict(max_trials=0), (1, "")),
    (dict(confidence=100.0), (1, "")),
    (dict(keypoints=False), (1, "")),
    (dict(out=False), (1, "")),
    (dict(one=True, method=9), (9, "")),
    (dict(one=True, keypoints=False), (1, "")),
])
def test_argument_errors_come_before_the_context(aps, case, want):
    assert _call(_library(aps), **case) == want


def test_argument_errors_come_in_order(aps):
    L = _library(aps)
    # the pairwise statuses first, then the RANSAC parameters, then keypoints, then out
    assert _call(L, dtype=7, max_trials=0, keypoints=False, out=False)[0] == 2
    assert _call(L, D=0, max_trials=0, keypoints=False, out=False)[0] == 4
    for case, word in ((dict(max_trials=0, keypoints=False, out=False), "max_trials"),
                       (dict(keypoints=False, out=False), "keypoints"), (dict(out=False), "out")):
        assert _call(L, **case)[0] == 1 and word in L.aps_last_error().decode(), case


def test_well_formed_calls_without_gpu_are_nogpu(aps):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by tests/test_gpu_pairwise_image_matching.py")
    L = _library(aps)
    assert _call(L) == (6, "apsmatch:nogpu")
    assert _call(L, one=True) == (6, "apsmatch:nogpu")
    assert _call(L, nsets=0, set_images=()) == (6, "apsmatch:nogpu")
    assert _call(L, rows=0, keypoints=False) == (6, "apsmatch:nogpu")   # no rows: keypoints are not needed
    assert _call(L, nsets=1, set_images=(2,), method=0, subset=400, rows=(1 << 30) - 600) == (6, "apsmatch:nogpu")
    d = [np.ones((3, 4), np.float32)] * 2
    kp = [np.zeros((3, 2))] * 2
    with pytest.raises(aps.ApsError) as e:
        aps.pairwiseImageMatchingSets(INP, [d], [2], [kp])
    assert e.value.identifier == "apsmatch:nogpu"
    with pytest.raises(aps.ApsError) as e:
        aps.pairwiseImageMatching(INP, d, 2, kp)
    assert e.value.identifier == "apsmatch:nogpu"


def test_host_mirror_guards(aps):
    d = [np.ones((3, 4), np.float32)] * 2
    kp = [np.zeros((3, 2))] * 2
    for field in (dict(imageMatchingMethod="mlesac"), dict(useMATLABImageMatching=1), dict(transformationType="affine"),
                  dict(apsGPUs=[1]), dict(Matchingmethod="fancy"),
                  dict(Matchingmethod="Approximate", ApproxFloatNNMethod="lsh")):
        with pytest.raises(ValueError):
            aps.pairwiseImageMatchingSets(dict(INP, **field), [d], [2], [kp])
        with pytest.raises(ValueError):
            aps.pairwiseImageMatching(dict(INP, **field), d, 2, kp)
    with pytest.raises(ValueError, match="numImgs"):
        aps.pairwiseImageMatchingSets(INP, [d], [0], [kp])
    with pytest.raises(ValueError, match="one keypoint set"):
        aps.pairwiseImageMatchingSets(INP, [d], [2], [kp, kp])
    with pytest.raises(ValueError, match="one per image"):
        aps.pairwiseImageMatchingSets(INP, [d], [2], [kp[:1]])
    with pytest.raises(ValueError, match="one row per descriptor"):
        aps.pairwiseImageMatchingSets(INP, [d], [2], [[np.zeros((2, 2)), kp[1]]])
    with pytest.raises(ValueError, match="numImg"):
        aps.pairwiseImageMatching(INP, d, 0, kp)


def test_semantics_warning(aps):
    d = [np.ones((3, 4), np.float32)] * 2
    kp = [np.zeros((3, 2))] * 2
    with pytest.warns(aps.ApsSemanticsWarning):
        try:
            aps.pairwiseImageMatchingSets(dict(INP, useMATLABFeatureMatch=1), [d], [2], [kp])
        except aps.ApsError as e:   # no GPU
            assert e.identifier == "apsmatch:nogpu"


def test_gateway_argument_checks(aps):
    import torch

    _library(aps)
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    args = ["gpu"] if torch.cuda.is_available() else []
    for gate in ("gate_pimatch", "gate_gimatch"):
        r = subprocess.run([os.path.join(ROOT, "mex", "_build", gate)] + args, capture_output=True, text=True)
        assert r.returncode == 0 and "OK" in r.stdout, gate + r.stdout + r.stderr


def test_new_kernels_compile_without_spills(tmp_path):
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
    for kernel in ("k_scatter_counts", "k_place_rows"):
        hits = [v for n, v in found.items() if kernel in n]
        assert hits, (kernel, sorted(found))
        assert all(v == (0, 0, 0) for v in hits), (kernel, hits)
