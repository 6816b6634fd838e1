"""imageMatching over many image sets in one call (aps_select_partners_sets, aps_image_matching_sets) without a GPU:
arguments are checked before any device is touched and carry the single-set entries' ids, a well-formed call fails with
apsmatch:nogpu (no CPU fallback), the host mirror rejects input.apsGPUs, malformed numImgs, non n x n cells and other
models than 'ransac' / 'projective', and the gateway aps_imageMatchingSets_mex checks its arguments under the mex shim."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INP = {"maxDistance": 5.5, "inliersConfidence": 99.9, "maxIter": 500, "mBrownLowe": 6}


def _library(aps):
    if not os.path.exists(aps.library_path()):
        pytest.skip("libapsmatch.so not built")
    return aps._lib.lib()


def _no_gpu(aps):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present: covered by tests/test_gpu_image_matching_sets.py")
    return _library(aps)


def _select(L, nsets, set_images, counts, spp=True):
    si = (C.c_int * max(len(set_images), 1))(*set_images)
    cnt = (C.c_int64 * max(len(counts), 1))(*counts)
    cand = (C.c_uint8 * max(len(counts), 1))()
    lin = (C.c_int64 * max(len(counts), 1))()
    out = (C.c_int64 * (max(nsets, 0) + 1))()
    return L.aps_select_partners_sets(None, nsets, si, cnt, 4, cand, lin, out if spp else None)


def _two_sets(bad_row=None, bad_lin=None):
    """set 1: two images, 4 correspondences in cell (1,2); set 2: two images, 5 correspondences"""
    pp = [np.array([0, 0, 0, 4, 4], np.int64), np.array([0, 0, 0, 5, 5], np.int64)]
    rows = [np.tile(np.array([1, 1], np.uint32), 4), np.tile(np.array([2, 3], np.uint32), 5)]
    if bad_row is not None:
        rows[1][bad_row] = 7     # image 2 of set 2 has 6 keypoints, image 1 has 3
    kp = np.zeros((3 + 3 + 3 + 6, 2))
    img_off = np.array([0, 3, 6, 9, 15], np.int64)
    spp = np.array([0, 1, 2], np.int64)
    lin = np.array([2, 2 if bad_lin is None else bad_lin], np.int64)
    return pp, rows, kp, img_off, spp, lin


def _match(L, nsets=2, set_images=(2, 2), args=None, ctx=None):
    pp, rows, kp, img_off, spp, lin = args or _two_sets()
    B = max(len(set_images), 1)
    si = (C.c_int * B)(*set_images)
    ppa = (C.c_void_p * B)(*[p.ctypes.data for p in pp][:B])
    ra = (C.c_void_p * B)(*[r.ctypes.data for r in rows][:B])
    P, T = int(spp[-1]), 9
    ptr, models, minv = np.zeros(P + 1, np.int64), np.zeros(9 * P), np.zeros(9 * P)
    inl, ni, acc, du = np.zeros(T, np.uint8), np.zeros(P, np.int32), np.zeros(P, np.uint8), np.zeros(P, np.int32)
    v = lambda a: C.c_void_p(a.ctypes.data)  # noqa: E731
    rc = L.aps_image_matching_sets(ctx, nsets, si, ppa, ra, v(kp), v(img_off), v(spp), v(lin), 5.5, 99.9, 500, None,
                                   1000, 0, v(ptr), v(models), v(minv), v(inl), v(ni), v(acc), v(du))
    return rc, L.aps_error_id().decode(), L.aps_last_error().decode(), ptr


def test_symbols_are_declared_and_bound(aps):
    L = _library(aps)
    hdr = open(os.path.join(ROOT, "include", "apsmatch.h")).read()
    for sym in ("aps_select_partners_sets", "aps_image_matching_sets"):
        assert sym in L._aps_symbols and sym in hdr
    assert "imageMatchingSets" in dir(aps) and "selectImagePartnersSets" in dir(aps)


@pytest.mark.parametrize("case", [
    dict(nsets=-1, set_images=[], counts=[]),
    dict(nsets=2, set_images=[1, -1], counts=[0]),
    dict(nsets=1, set_images=[2], counts=[0, 1, 1, 0], spp=False),
])
def test_select_partners_sets_argument_errors(aps, case):
    L = _library(aps)
    assert _select(L, **case) == 1               # APS_ERR_ARGS, before the (missing) context
    assert L.aps_error_id().decode() == ""


def test_image_matching_sets_argument_errors(aps):
    L = _library(aps)
    assert _match(L, nsets=-1, set_images=())[0] == 1
    assert _match(L, set_images=(2, -2))[0] == 1
    rc, eid, msg, _ = _match(L, args=_two_sets(bad_lin=4))      # cell index outside set 2's 2 x 2 block
    assert (rc, eid) == (1, "") and "set 2" in msg
    rc, eid, msg, ptr = _match(L, args=_two_sets(bad_row=3))    # row 2 of set 2's cell: index 7 > 6 keypoints
    assert (rc, eid) == (1, "refineMatch:MatchIndexOutOfBounds") and "set 2" in msg
    assert not ptr.any()                                         # the call returns nothing
    rc, eid, _, _ = _match(L, args=_two_sets(bad_row=0))        # 7 > 3 keypoints of image 1
    assert eid == "refineMatch:MatchIndexOutOfBounds"


def test_well_formed_calls_without_gpu_are_nogpu(aps):
    L = _no_gpu(aps)
    assert _select(L, 2, [2, 0], [0, 3, 3, 0]) == 6              # APS_ERR_NOGPU
    assert L.aps_error_id().decode() == "apsmatch:nogpu"
    assert _select(L, 0, [], []) == 6
    rc, eid, _, _ = _match(L)
    assert (rc, eid) == (6, "apsmatch:nogpu")
    kps = [np.zeros((5, 2)), np.zeros((5, 2))]
    m = [[np.zeros((0, 0)), np.ones((4, 2))], [np.zeros((0, 0))] * 2]
    with pytest.raises(aps.ApsError) as e:
        aps.imageMatchingSets(INP, [2, 2], [kps, kps], [m, m])
    assert e.value.identifier == "apsmatch:nogpu"


def test_host_mirror_rejects_malformed_input(aps):
    kps = [np.zeros((5, 2)), np.zeros((5, 2))]
    m = [[np.zeros((0, 0)), np.ones((4, 2))], [np.zeros((0, 0))] * 2]
    with pytest.raises(ValueError, match="apsGPUs"):
        aps.imageMatchingSets(dict(INP, apsGPUs=[1]), [2, 2], [kps, kps], [m, m])
    for bad in ([2], [2, -1], [2, 1.5], [2, float("nan")], [2, 2, 2]):
        with pytest.raises(ValueError, match="numImgs"):
            aps.imageMatchingSets(INP, bad, [kps, kps], [m, m])
    with pytest.raises(ValueError, match="n-by-n"):
        aps.imageMatchingSets(INP, [2, 2], [kps, kps], [m, [m[0]]])
    with pytest.raises(ValueError, match="n-by-n"):
        aps.imageMatchingSets(INP, [2, 3], [kps, kps + kps[:1]], [m, m])
    with pytest.raises(ValueError, match="one per image"):
        aps.imageMatchingSets(INP, [2, 2], [kps, kps[:1]], [m, m])
    for field in (dict(imageMatchingMethod="mlesac"), dict(useMATLABImageMatching=1),
                  dict(transformationType="affine")):
        with pytest.raises(ValueError):
            aps.imageMatchingSets(dict(INP, **field), [2, 2], [kps, kps], [m, m])


def test_gateway_argument_checks(aps):
    import torch

    _library(aps)
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    args = ["gpu"] if torch.cuda.is_available() else []
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_imatch_sets")] + args, capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
