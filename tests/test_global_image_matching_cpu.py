"""featureMatchingGlobal + imageMatching in one call (aps_global_image_matching[_sets]) without a GPU: argument errors
are raised before any device is touched and carry the ids of aps_feature_matching_global_sets, a well-formed call fails
with apsmatch:nogpu (no CPU fallback), the host mirror rejects 'mlesac', non-projective models and input.apsGPUs, the
gateway aps_globalImageMatching_mex checks its arguments under the mex shim, and the new kernels compile for sm_100a
without local-memory spills."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "automaticpanoramicimagestitching-autopanostitch-matlab_b200", "csrc")
INP = {"k": 4, "Ratiothreshold": 0.8, "maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}


def _library(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    return aps._lib.lib()


def _call(L, nsets=2, set_images=(2, 1), D=4, dtype=0, k=4, max_trials=500, confidence=99.9, keypoints=True,
          out=True, one=False):
    counts = [3] * max(sum(max(s, 0) for s in set_images), 1)
    desc = np.zeros((3, max(D, 1)), np.float32)
    ptrs = (C.c_void_p * len(counts))(*([desc.ctypes.data] * len(counts)))
    cnt = (C.c_int64 * len(counts))(*counts)
    kp = np.zeros((3 * len(counts), 2))
    h = C.c_void_p()
    tail = (C.c_void_p(kp.ctypes.data) if keypoints else None, 6, 5.5, confidence, max_trials, 0, 0,
            C.byref(h) if out else None)
    if one:
        rc = L.aps_global_image_matching(None, ptrs, cnt, set_images[0], D, dtype, 1, k, 0.8, 0, 0, *tail)
    else:
        si = (C.c_int * max(len(set_images), 1))(*set_images)
        rc = L.aps_global_image_matching_sets(None, nsets, si, ptrs, cnt, D, dtype, 1, k, 0.8, 0, 0, *tail)
    return rc, L.aps_error_id().decode()


def test_symbols_are_declared_and_bound(aps):
    L = _library(aps)
    hdr = open(os.path.join(ROOT, "include", "apsmatch.h")).read()
    for sym in ("aps_global_image_matching_sets", "aps_global_image_matching", "aps_image_matches_free"):
        assert sym in L._aps_symbols and sym in hdr
    assert L.aps_abi_version() == 1
    assert "globalImageMatchingSets" in dir(aps) and "globalImageMatching" in dir(aps)


@pytest.mark.parametrize("case, want", [
    (dict(nsets=-1, set_images=()), (1, "")),
    (dict(set_images=(2, -1)), (1, "")),
    (dict(k=0), (3, "flann_knn:k")),
    (dict(k=33), (3, "flann_knn:k")),
    (dict(dtype=7), (2, "flann_knn:type")),
    (dict(D=0), (4, "flann_knn:dim")),
    (dict(max_trials=0), (1, "")),
    (dict(confidence=100.0), (1, "")),
    (dict(keypoints=False), (1, "")),
    (dict(out=False), (1, "")),
    (dict(one=True, k=0), (3, "flann_knn:k")),
    (dict(one=True, keypoints=False), (1, "")),
])
def test_argument_errors_come_before_the_context(aps, case, want):
    assert _call(_library(aps), **case) == want


def test_well_formed_calls_without_gpu_are_nogpu(aps):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by tests/test_gpu_global_image_matching.py")
    L = _library(aps)
    assert _call(L) == (6, "apsmatch:nogpu")
    assert _call(L, one=True) == (6, "apsmatch:nogpu")
    assert _call(L, nsets=0, set_images=()) == (6, "apsmatch:nogpu")
    d = [np.ones((3, 4), np.float32)] * 2
    kp = [np.zeros((3, 2))] * 2
    with pytest.raises(aps.ApsError) as e:
        aps.globalImageMatchingSets(INP, [d], [2], [kp])
    assert e.value.identifier == "apsmatch:nogpu"


def test_host_mirror_guards(aps):
    d = [np.ones((3, 4), np.float32)] * 2
    kp = [np.zeros((3, 2))] * 2
    for field in (dict(imageMatchingMethod="mlesac"), dict(useMATLABImageMatching=1), dict(transformationType="affine"),
                  dict(apsGPUs=[1])):
        with pytest.raises(ValueError):
            aps.globalImageMatchingSets(dict(INP, **field), [d], [2], [kp])
        with pytest.raises(ValueError):
            aps.globalImageMatching(dict(INP, **field), d, 2, kp)
    with pytest.raises(ValueError, match="numImgs"):
        aps.globalImageMatchingSets(INP, [d], [0], [kp])
    with pytest.raises(ValueError, match="one keypoint set"):
        aps.globalImageMatchingSets(INP, [d], [2], [kp, kp])
    with pytest.raises(ValueError, match="one per image"):
        aps.globalImageMatchingSets(INP, [d], [2], [kp[:1]])
    with pytest.raises(ValueError, match="one row per descriptor"):
        aps.globalImageMatchingSets(INP, [d], [2], [[np.zeros((2, 2)), kp[1]]])
    with pytest.raises(ValueError, match="numImg"):
        aps.globalImageMatching(INP, d, 0, kp)


def test_gateway_argument_checks(aps):
    import torch

    _library(aps)
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    args = ["gpu"] if torch.cuda.is_available() else []
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_gimatch")] + args, capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr


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
    for kernel in ("k_candidate_tables", "k_scan_countsINS_7CountOf", "k_scan_countsINS_15AcceptedInliers",
                   "k_pack_rows", "k_all_matches"):
        hits = [v for n, v in found.items() if kernel in n]
        assert hits, (kernel, sorted(found))
        assert all(v == (0, 0, 0) for v in hits), (kernel, hits)
