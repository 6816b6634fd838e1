"""Device groups on the GPU: the one-call global and pairwise entries spread over several GPUs of this process return
lists BIT-IDENTICAL to the single-context calls (pair_ptr, rows, metric), and match the oracle where it is cheap.  The
per-member statistics prove that the work was spread.  Multi-device cases skip with fewer than 2 visible GPUs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ndev():
    import torch

    return torch.cuda.device_count()


def _multi():
    n = _ndev()
    if n < 2:
        pytest.skip("needs at least 2 visible GPUs")
    return list(range(min(n, 8)))


_shared = {}


@pytest.fixture(params=["gpus", "shared3", "shared8"])
def group(request, aps):
    """A group over the visible GPUs (skipped with fewer than 2), and groups of 3 and 8 members sharing GPU 0 -- the
    same multi-member pipeline, runnable on a one-GPU machine."""
    if request.param == "gpus":
        return aps._lib.default_group(_multi())
    m = int(request.param[6:])
    if m not in _shared:
        _shared[m] = aps.DeviceGroup([0], shared_members=m)
    return _shared[m]


def _args(aps, desc, fortran=False):
    host = aps.host
    mats = [None if d is None or len(d) == 0 else (np.asfortranarray(d) if fortran else np.ascontiguousarray(d))
            for d in desc]
    counts = [0 if m is None else m.shape[0] for m in mats]
    ptrs, cnt, layout, keep = host._desc_args(mats, counts)
    D = next(m.shape[1] for m in mats if m is not None)
    return ptrs, cnt, layout, keep, D


def _csr(aps, h, n):
    try:
        return aps.host._csr_from_matchlist(h, n)
    finally:
        aps._lib.lib().aps_matchlist_free(h)


def global_single(aps, desc, k, ratio, binary=False, fortran=False):
    ptrs, cnt, layout, keep, D = _args(aps, desc, fortran)
    h = C.c_void_p()
    aps._lib.check(aps._lib.lib().aps_feature_matching_global(aps._lib.default_context().handle, ptrs, cnt, len(desc), D,
                                                              int(binary), layout, k, ratio, 0, C.byref(h)))
    return _csr(aps, h, len(desc))


def global_group(aps, group, desc, k, ratio, binary=False, fortran=False, mutual=0):
    ptrs, cnt, layout, keep, D = _args(aps, desc, fortran)
    h = C.c_void_p()
    aps._lib.check(aps._lib.lib().aps_group_feature_matching_global(group.handle, ptrs, cnt, len(desc), D, int(binary),
                                                                    layout, k, ratio, mutual, C.byref(h)))
    return _csr(aps, h, len(desc))


def pairwise_single(aps, desc, thr, ratio, method=0, subset=12000, seed=0, binary=False):
    """The single-context call of the host mirror (aps_feature_matching_pairwise_shard, or the staged plan with the
    method for 'Approximate')."""
    names = {0: "Exhaustive", 1: "subsetpdist2", 2: "kdtree", 3: "pca2nn"}
    inp = {"Matchingthreshold": thr, "Ratiothreshold": ratio, "apsSubset": subset, "apsSeed": seed,
           "Matchingmethod": "Exhaustive" if method == 0 else "Approximate", "ApproxFloatNNMethod": names[method]}
    cells = [aps.binaryFeatures(d) for d in desc] if binary else desc
    return aps.featureMatchingPairwise(inp, cells, len(desc), csr=True)


def pairwise_group(aps, group, desc, thr, ratio, method=0, subset=12000, seed=0, binary=False):
    ptrs, cnt, layout, keep, D = _args(aps, desc)
    h = C.c_void_p()
    aps._lib.check(aps._lib.lib().aps_group_feature_matching_pairwise(group.handle, ptrs, cnt, len(desc), D, int(binary),
                                                                      layout, thr, ratio, method, subset, seed,
                                                                      C.byref(h)))
    return _csr(aps, h, len(desc))


def assert_same(a, b):
    assert a[0].dtype == b[0].dtype and np.array_equal(a[0], b[0]), "pair_ptr"
    assert a[1].dtype == b[1].dtype and np.array_equal(a[1], b[1]), "rows"
    assert a[2].tobytes() == b[2].tobytes(), "metric"


def assert_oracle(csr, ref_cells, n):
    pp, rows = csr[0], csr[1]
    for j in range(n):
        for i in range(j):
            c = i + j * n
            got = rows[pp[c]:pp[c + 1]].astype(np.float64)
            exp = ref_cells.get((i, j))
            if exp is None or len(exp) == 0:
                assert len(got) == 0, (i, j)
            else:
                assert got.shape == exp.shape and (got == exp).all(), (i, j)


def assert_rows_spread(aps, group, F):
    bounds = aps.multigpu.shard_bounds(F, len(group))
    for i, (q0, q1) in enumerate(bounds):
        assert group.ctx(i).last_stats()["rows"] == q1 - q0, (i, q0, q1)


# ---- global ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [4, 8])
def test_global_c2_equals_single_context(aps, k, group):
    desc, c = aps.synth.make_config(2)
    one = global_single(aps, desc, k, c["ratio"])
    grp = global_group(aps, group, desc, k, c["ratio"])
    assert_same(grp, one)
    assert grp[1].shape[0] > 0
    assert_rows_spread(aps, group, sum(len(d) for d in desc))


def test_global_mutual_equals_single_context(aps, orc, group):
    desc, c = aps.synth.make_config(1, n=6, kp=2048)
    inp = {"k": c["k"], "Ratiothreshold": c["ratio"], "apsMutual": 1}
    one = aps.featureMatchingGlobal(inp, desc, len(desc))
    distinct = len(set(group.devices)) == len(group)
    grp_cells = (aps.featureMatchingGlobal(dict(inp, apsGPUs=[d + 1 for d in group.devices]), desc, len(desc))
                 if distinct else one)
    csr = global_group(aps, group, desc, c["k"], c["ratio"], mutual=1)
    n = len(desc)
    for j in range(n):
        for i in range(j):
            assert np.array_equal(grp_cells[i][j], one[i][j]), (i, j)
            cc = i + j * n
            assert np.array_equal(csr[1][csr[0][cc]:csr[0][cc + 1]].astype(np.float64).reshape(-1, 2),
                                  np.asarray(one[i][j]).reshape(-1, 2)), (i, j)
    # the cross-check only removes rows
    plain = global_group(aps, group, desc, c["k"], c["ratio"])
    assert csr[1].shape[0] <= plain[1].shape[0]


def test_global_binary_equals_single_context_and_oracle(aps, orc, group):
    desc, c = aps.synth.make_config(4, n=6, kp=3000)
    one = global_single(aps, desc, c["k"], c["ratio"], binary=True)
    grp = global_group(aps, group, desc, c["k"], c["ratio"], binary=True)
    assert_same(grp, one)
    assert_oracle(grp, orc.feature_matching_global(desc, c["k"], c["ratio"])["cells"], len(desc))
    assert_rows_spread(aps, group, sum(len(d) for d in desc))


def test_global_fewer_rows_than_members(aps, orc, group):
    """F = 100 < 128: member 0 searches everything, every other member gets an empty block."""
    rng = np.random.default_rng(11)
    base = rng.integers(0, 200, (40, 128)).astype(np.float32)
    desc = [base, np.zeros((0, 128), np.float32), base[:30] + rng.integers(0, 3, (30, 128)).astype(np.float32),
            base[10:40] + 1]
    one = global_single(aps, desc, 4, 0.8)
    grp = global_group(aps, group, desc, 4, 0.8)
    assert_same(grp, one)
    assert grp[1].shape[0] > 0
    assert_oracle(grp, orc.feature_matching_global([d for d in desc], 4, 0.8)["cells"], len(desc))
    assert_rows_spread(aps, group, 100)


def test_global_empty_images_and_cut_images_col_major(aps, orc, group):
    """Empty images, images that straddle 128-row block boundaries, and column-major (MATLAB) input."""
    desc, c = aps.synth.make_config(1, n=8, kp=1000)
    sizes = [301, 0, 517, 0, 1000, 77, 600, 0]
    desc = [d[:s] for d, s in zip(desc, sizes)]
    one = global_single(aps, desc, c["k"], c["ratio"])
    grp = global_group(aps, group, desc, c["k"], c["ratio"], fortran=True)
    assert_same(grp, one)
    assert_oracle(grp, orc.feature_matching_global(desc, c["k"], c["ratio"])["cells"], len(desc))
    assert_rows_spread(aps, group, sum(sizes))


def test_global_all_empty(aps, group):
    desc = [np.zeros((0, 128), np.float32), np.zeros((0, 128), np.float32)]
    ptrs, cnt, layout, keep = aps.host._desc_args([None, None], [0, 0])
    h = C.c_void_p()
    aps._lib.check(aps._lib.lib().aps_group_feature_matching_global(group.handle, ptrs, cnt, 2, 128, 0, layout, 4, 0.8, 0,
                                                                    C.byref(h)))
    pp, rows, _ = _csr(aps, h, len(desc))
    assert (pp == 0).all() and rows.shape[0] == 0


# ---- pairwise ----------------------------------------------------------------------------------------------------
def _pairs_with_share(counts, n, N):
    share = [0] * N
    o = 0
    for j in range(n):
        for i in range(j):
            if counts[i] and counts[j]:
                share[o % N] += 1
            o += 1
    return share


def test_pairwise_exhaustive_equals_single_context_and_oracle(aps, orc, group):
    desc, c = aps.synth.make_config(5, n=12, kp=1024)
    desc[4] = desc[4][:0]
    one = pairwise_single(aps, desc, 1.5, 0.7)
    single_screened = aps._lib.default_context().pairwise_stats()["pairs_screened"]
    grp = pairwise_group(aps, group, desc, 1.5, 0.7)
    assert_same(grp, one)
    assert grp[1].shape[0] > 0
    ref = orc.feature_matching_pairwise(desc, 1.5, 0.7)
    assert_oracle(grp, ref["cells"] if isinstance(ref, dict) else ref, len(desc))
    screened = [group.ctx(i).pairwise_stats()["pairs_screened"] for i in range(len(group))]
    assert sum(screened) == single_screened
    share = _pairs_with_share([len(d) for d in desc], len(desc), len(group))
    for s, got in zip(share, screened):
        assert s == 0 or got > 0, (share, screened)


@pytest.mark.parametrize("method", [1, 2, 3])
def test_pairwise_approximate_methods_equal_single_context(aps, method, group):
    """'subsetpdist2' (image 2 above the subset size, so it is searched through its subset view), 'kdtree', 'pca2nn'."""
    desc, c = aps.synth.make_config(5, n=8, kp=700)
    desc[2] = np.vstack([desc[2], desc[3][:500]])
    one = pairwise_single(aps, desc, 1.5, 0.7, method=method, subset=900, seed=7)
    grp = pairwise_group(aps, group, desc, 1.5, 0.7, method=method, subset=900, seed=7)
    assert_same(grp, one)
    assert grp[1].shape[0] > 0


def test_pairwise_binary_equals_single_context(aps, group):
    desc, c = aps.synth.make_config(4, n=6, kp=1500)
    one = pairwise_single(aps, desc, 40.0, 0.8, binary=True)
    grp = pairwise_group(aps, group, desc, 40.0, 0.8, binary=True)
    assert_same(grp, one)


def test_pairwise_more_members_than_pairs(aps, orc, group):
    desc, c = aps.synth.make_config(5, n=2, kp=800)
    one = pairwise_single(aps, desc, 1.5, 0.7)
    grp = pairwise_group(aps, group, desc, 1.5, 0.7)
    assert_same(grp, one)
    ref = orc.feature_matching_pairwise(desc, 1.5, 0.7)
    assert_oracle(grp, ref["cells"] if isinstance(ref, dict) else ref, 2)


def test_host_mirror_apsGPUs(aps):
    devs = _multi()
    desc, c = aps.synth.make_config(5, n=6, kp=600)
    inp = {"Matchingmethod": "Exhaustive", "Matchingthreshold": 1.5, "Ratiothreshold": 0.7}
    one = aps.featureMatchingPairwise(inp, desc, len(desc))
    grp = aps.featureMatchingPairwise(dict(inp, apsGPUs=[d + 1 for d in devs]), desc, len(desc))
    for j in range(len(desc)):
        for i in range(j):
            assert grp[i][j].shape == one[i][j].shape and (grp[i][j] == one[i][j]).all()


def test_stage_times_are_reported(aps, group):
    desc, c = aps.synth.make_config(1, n=6, kp=2048)
    global_group(aps, group, desc, c["k"], c["ratio"])
    t0 = group.stage_times(0)
    assert t0["upload"] > 0 and t0["search"] > 0 and t0["finish"] > 0
    for i in range(1, len(group)):
        assert group.stage_times(i)["finish"] == 0.0


# ---- one member, argument checks (any GPU count) ------------------------------------------------------------------
def test_one_member_group_equals_plain_entries(aps):
    group = aps.DeviceGroup([0])
    try:
        desc, c = aps.synth.make_config(1, n=5, kp=1500)
        assert_same(global_group(aps, group, desc, c["k"], c["ratio"]), global_single(aps, desc, c["k"], c["ratio"]))
        kz, _ = aps.synth.make_config(5, n=5, kp=700)
        assert_same(pairwise_group(aps, group, kz, 1.5, 0.7), pairwise_single(aps, kz, 1.5, 0.7))
        assert_same(pairwise_group(aps, group, kz, 1.5, 0.7, method=3), pairwise_single(aps, kz, 1.5, 0.7, method=3))
        assert group.ctx(0).last_stats()["rows"] >= 0
    finally:
        group.close()


@pytest.mark.parametrize("devices", [[0, 0], [0, 4096], [-1], []])
def test_bad_device_lists_are_args_errors(aps, devices):
    with pytest.raises(aps.ApsError) as e:
        aps.DeviceGroup(devices)
    assert e.value.code == 1


def _run_gate_gpus(mats, scalars, gpus, tmp_path, error_id=None):
    """File mode of mex/shim_driver.cpp (as tests/test_mex_gateways.py drives it) with the trailing device list.
    error_id: the call must fail with that MATLAB error identifier instead."""
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    with open(fin, "wb") as f:
        f.write(np.int32(len(mats)).tobytes())
        for cls, a in mats:
            f.write(np.array([cls, a.shape[0], a.shape[1]], np.int32).tobytes())
            f.write(np.asfortranarray(a).tobytes(order="F"))
        f.write(np.int32(len(scalars)).tobytes())
        f.write(np.asarray(scalars, np.float64).tobytes())
        f.write(np.int32(len(gpus)).tobytes())
        f.write(np.asarray(gpus, np.float64).tobytes())
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_batched"), "file", fin, fout], capture_output=True,
                       text=True)
    if error_id is not None:
        assert r.returncode == 1 and f"ERROR {error_id}:" in r.stdout, r.stdout + r.stderr
        return None
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
    raw = open(fout, "rb").read()
    pos, outs = 4, []
    for _ in range(int(np.frombuffer(raw, np.int32, 1)[0])):
        cls, rows, cols = (int(v) for v in np.frombuffer(raw, np.int32, 3, pos))
        pos += 12
        if cls < 0:
            outs.append(None)
            continue
        assert cls == 2
        outs.append(np.frombuffer(raw, np.float64, rows * cols, pos).reshape((rows, cols), order="F"))
        pos += rows * cols * 8
    return outs


def _gate_cells_equal(outs, ref_cells, n):
    o = 0
    for j in range(n):
        for i in range(j):
            exp, got = ref_cells.get((i, j)), outs[o]
            o += 1
            if exp is None or len(exp) == 0:
                assert got is None or got.shape[0] == 0, (i, j)
            else:
                assert got is not None and got.shape == exp.shape and (got == exp).all(), (i, j)


def test_gateway_with_device_list_matches_the_oracle(aps, orc, tmp_path):
    gpus = [d + 1 for d in _multi()]
    desc, c = aps.synth.make_config(1, n=4, kp=700)
    outs = _run_gate_gpus([(0, d) for d in desc], [0, c["k"], c["ratio"], 0], gpus, tmp_path)
    _gate_cells_equal(outs, orc.feature_matching_global(desc, c["k"], c["ratio"])["cells"], len(desc))
    kz, _ = aps.synth.make_config(5, n=5, kp=500)
    outs = _run_gate_gpus([(0, d) for d in kz], [1, 1.5, 0.6, 0], gpus, tmp_path)
    ref = orc.feature_matching_pairwise(kz, 1.5, 0.6)
    _gate_cells_equal(outs, ref["cells"] if isinstance(ref, dict) else ref, len(kz))


def test_gateway_gpu_that_does_not_exist_is_an_args_error(aps, tmp_path):
    """A list naming a GPU beyond the visible ones (MATLAB numbering) raises apsmatch:args, not apsmatch:nogpu."""
    desc, c = aps.synth.make_config(1, n=3, kp=300)
    for mode, scalars in ((0, [0, c["k"], c["ratio"], 0]), (1, [1, 1.5, 0.6, 0])):
        _run_gate_gpus([(0, d) for d in desc], scalars, [1, _ndev() + 1], tmp_path, error_id="apsmatch:args")
