"""featureMatchingGlobal over many independent image sets in one call (aps_feature_matching_global_sets): every set's
match list is bit-identical to featureMatchingGlobal on that set alone (and to the oracle where that is cheap), rows of
one set never see another set's rows, and the pooled pass's launch count does not grow with the number of sets."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(aps):
    return aps._lib.default_context()


def _same_cells(got, exp, n):
    """bit-for-bit: same cell sizes (pair_ptr) and same rows; returns the number of match rows"""
    rows = 0
    assert len(got) == n and len(exp) == n
    for i in range(n):
        for j in range(n):
            g, e = np.asarray(got[i][j]), np.asarray(exp[i][j])
            assert g.shape == e.shape, (i, j, g.shape, e.shape)
            assert g.dtype == e.dtype and np.array_equal(g, e), (i, j)
            rows += g.shape[0] if g.ndim == 2 else 0
    return rows


def _oracle_equal(orc, got, desc, k, ratio):
    ref = orc.feature_matching_global(desc, k, ratio)
    n = len(desc)
    for i in range(n):
        for j in range(n):
            e = ref["cells"].get((i, j)) if i < j else None
            g = got[i][j]
            if e is None:
                assert g.size == 0, (i, j)
            else:
                assert g.shape == e.shape and (g == e).all(), (i, j)


def _check_sets(aps, sets, inp, ctx, orc=None):
    """the batched call against featureMatchingGlobal per set; returns the total match rows"""
    nums = [len(s) for s in sets]
    got = aps.featureMatchingGlobalSets(inp, sets, nums, ctx=ctx)
    assert len(got) == len(sets)
    rows = 0
    for b, s in enumerate(sets):
        single = aps.featureMatchingGlobal(inp, s, nums[b], ctx=ctx)
        rows += _same_cells(got[b], single, nums[b])
        if orc is not None and not inp.get("apsMutual") and any(np.asarray(getattr(x, "Features", x)).shape[0] for x in s):
            raw = [x.Features if isinstance(x, aps.binaryFeatures) else x for x in s]
            _oracle_equal(orc, got[b], raw, inp["k"], inp["Ratiothreshold"])
    return got, rows


def _sift_images(aps, counts, seed, D=128, kind="sift"):
    """len(counts) images with planted overlaps, image i cut to counts[i] rows"""
    kp = max(300, max(counts))
    imgs = aps.synth.synth_descriptors(kind, len(counts), kp, D, seed)
    return [np.ascontiguousarray(im[:c]) for im, c in zip(imgs, counts)]


# set shapes: sizes that are not multiples of 128, a single image, all images empty, an empty image inside a set,
# fewer than k + 1 rows, and a set whose rows are all identical
SHAPES = [[173, 300, 251], [300], [0, 0], [200, 0, 150, 99], [2, 1], "identical", [300, 300]]


def _mixed_sets(aps, kind, D):
    sets = []
    for b, sh in enumerate(SHAPES):
        if sh == "identical":
            row = _sift_images(aps, [1], 900 + b, D, kind)[0]
            sets.append([np.repeat(row, 20, axis=0) for _ in range(3)])
        else:
            sets.append(_sift_images(aps, sh, 700 + b, D, kind))
    return sets


@pytest.mark.parametrize("k", [4, 8, 12])
@pytest.mark.parametrize("mutual", [0, 1])
def test_float_sets_match_single_set_calls(aps, orc, ctx, k, mutual):
    sets = _mixed_sets(aps, "sift", 128)
    _, rows = _check_sets(aps, sets, {"k": k, "Ratiothreshold": 0.8, "apsMutual": mutual}, ctx, orc)
    assert rows > 100


# sets large enough for the tensor path (n_b^2 >= 2^22), sizes not multiples of the 256-row unit, mixed with small sets
TENSOR_SHAPES = [[1100, 1000, 333], [2048, 0, 2048, 700], [1500, 1500]]


@pytest.mark.parametrize("k", [4, 8, 12])
@pytest.mark.parametrize("mutual", [0, 1])
def test_tensor_sized_sets_in_one_pass(aps, ctx, k, mutual):
    """the tensor-path sets share ONE tcgen05 unit-table launch; the stats say so"""
    big = [_sift_images(aps, sh, 1700 + b) for b, sh in enumerate(TENSOR_SHAPES)]
    small = _mixed_sets(aps, "sift", 128)[:3]
    sets = [big[0], small[0], big[1], small[1], small[2], big[2]]
    _, rows = _check_sets(aps, sets, {"k": k, "Ratiothreshold": 0.8, "apsMutual": mutual}, ctx)
    aps.featureMatchingGlobalSets({"k": k, "Ratiothreshold": 0.8, "apsMutual": mutual}, sets, [len(x) for x in sets],
                                  ctx=ctx)
    st = ctx.last_stats()
    assert st["engine"] == "tcgen05" and st["rows"] == sum(m.shape[0] for x in sets for m in x)
    assert rows > 1000


def test_binary_sets_match_single_set_calls(aps, orc, ctx):
    sets = [[aps.binaryFeatures(m) for m in s] for s in _mixed_sets(aps, "orb", 32)]
    _, rows = _check_sets(aps, sets, {"k": 4, "Ratiothreshold": 0.8, "BFMatch": 1}, ctx, orc)
    assert rows > 100
    _check_sets(aps, sets, {"k": 4, "Ratiothreshold": 0.8, "BFMatch": 1, "apsMutual": 1}, ctx)


@pytest.mark.parametrize("binary", [False, True])
def test_sets_are_isolated(aps, ctx, binary):
    """set B holds exact copies of set A's rows: a search that leaked across sets would find them at distance 0"""
    kind, D = ("orb", 32) if binary else ("sift", 128)
    a = _sift_images(aps, [1300, 1280, 1260], 11, D, kind)   # float: tensor-path sets
    b = [a[0].copy(), a[1][:900].copy()] + _sift_images(aps, [1240], 12, D, kind)
    wrap = (lambda s: [aps.binaryFeatures(m) for m in s]) if binary else (lambda s: s)
    inp = {"k": 4, "Ratiothreshold": 0.8}
    got, _ = _check_sets(aps, [wrap(a), wrap(b)], inp, ctx)
    # within set B the copies do find each other (same image contents as A's images 0 and 1): the lists are not empty
    assert sum(np.asarray(got[1][i][j]).shape[0] for i in range(3) for j in range(3) if i < j) > 0


def test_skewed_batch(aps, ctx):
    """one C2-sized set with 50 tiny sets: its 640 units and the tiny sets' groups in one pass"""
    big, c = aps.synth.make_config(2)
    tiny = [_sift_images(aps, [120 + b, 90], 3000 + b) for b in range(50)]
    got, rows = _check_sets(aps, [big] + tiny, {"k": c["k"], "Ratiothreshold": c["ratio"]}, ctx)
    assert rows > 10000
    aps.featureMatchingGlobalSets({"k": c["k"], "Ratiothreshold": c["ratio"]}, [big] + tiny, [len(big)] + [2] * 50,
                                  ctx=ctx)
    assert ctx.last_stats()["engine"] == "tcgen05"


def test_many_tiny_sets(aps, ctx):
    sets = [_sift_images(aps, [200, 200, 200], 5000 + b) for b in range(300)]
    _, rows = _check_sets(aps, sets, {"k": 4, "Ratiothreshold": 0.8}, ctx)
    assert rows > 300


def test_real_valued_batch_fallback_and_exact_engine(aps, ctx):
    """synth config 6 (real-valued SIFT) cut into 8 sets: the proof fails on some rows, so the set-restricted exact
    fallback runs inside the batch; every list equals the exact engine's and the single-set call's"""
    desc, c = aps.synth.make_config(6)
    cuts = [0, 3, 6, 9, 12, 14, 16, 18, 20]
    sets = [desc[cuts[b]:cuts[b + 1]] for b in range(8)]
    inp = {"k": c["k"], "Ratiothreshold": c["ratio"]}
    got, rows = _check_sets(aps, sets, inp, ctx)
    assert rows > 10000
    got = aps.featureMatchingGlobalSets(inp, sets, [len(s) for s in sets], ctx=ctx)
    assert ctx.first_pass_unproven() > 0
    st = ctx.last_stats()
    assert st["engine"] == "tcgen05" and st["rows"] == sum(d.shape[0] for d in desc)
    assert st["fallback_rows"] == ctx.first_pass_unproven() and not st["bf16_exact_operands"]
    ctx.set_float_engine(1)
    try:
        exact = aps.featureMatchingGlobalSets(inp, sets, [len(s) for s in sets], ctx=ctx)
        assert ctx.last_stats()["engine"] == "exact"
    finally:
        ctx.set_float_engine(0)
    for b in range(8):
        _same_cells(got[b], exact[b], len(sets[b]))


@pytest.mark.parametrize("shape", [[150, 130], [1200, 1100], [2048, 2048, 0, 2048, 2048, 2048]],
                         ids=["small", "tensor", "C1"])
def test_launch_count_does_not_grow_with_the_number_of_sets(aps, ctx, shape):
    L = aps._lib.lib()
    inp = {"k": 4, "Ratiothreshold": 0.8}
    delta = {}
    for B in (2, 200):
        base = _sift_images(aps, shape, 8000)
        sets = [[m[np.random.default_rng(b).permutation(m.shape[0])] for m in base] for b in range(B)]
        n = len(shape)
        aps.featureMatchingGlobalSets(inp, sets, [n] * B, ctx=ctx)   # warm-up
        n0 = L.aps_launch_count()
        aps.featureMatchingGlobalSets(inp, sets, [n] * B, ctx=ctx)
        delta[B] = L.aps_launch_count() - n0
    assert 0 < delta[200] <= delta[2], delta


def test_one_set_call_is_the_single_set_call(aps, ctx):
    desc, c = aps.synth.make_config(1)
    inp = {"k": c["k"], "Ratiothreshold": c["ratio"]}
    got = aps.featureMatchingGlobalSets(inp, [desc], [len(desc)], ctx=ctx)
    assert _same_cells(got[0], aps.featureMatchingGlobal(inp, desc, len(desc), ctx=ctx), len(desc)) > 500


def test_column_major_input(aps, ctx):
    sets = [[np.asfortranarray(m) for m in s] for s in _mixed_sets(aps, "sift", 128)]
    _check_sets(aps, sets, {"k": 4, "Ratiothreshold": 0.8}, ctx)


# ---- the MEX verb through the shim driver, against the per-set 'global' verb --------------------------------------
def _run_gate(mats, scalars, tmp_path):
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "mex"), "shimcheck"], check=True, capture_output=True)
    fin, fout = str(tmp_path / "in.bin"), str(tmp_path / "out.bin")
    with open(fin, "wb") as f:
        f.write(np.int32(len(mats)).tobytes())
        for cls, a in mats:
            f.write(np.array([cls, a.shape[0], a.shape[1]], np.int32).tobytes())
            f.write(np.asfortranarray(a).tobytes(order="F"))
        f.write(np.int32(len(scalars)).tobytes())
        f.write(np.asarray(scalars, np.float64).tobytes())
    r = subprocess.run([os.path.join(ROOT, "mex", "_build", "gate_batched"), "file", fin, fout], capture_output=True,
                       text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
    raw = open(fout, "rb").read()
    nout, pos, outs = int(np.frombuffer(raw, np.int32, 1)[0]), 4, []
    for _ in range(nout):
        cls, m, n = np.frombuffer(raw, np.int32, 3, pos)
        pos += 12
        if cls < 0:
            outs.append(None)
            continue
        dt = {0: np.float32, 1: np.uint8, 2: np.float64, 3: np.uint32}[int(cls)]
        cnt = int(m) * int(n)
        outs.append(np.frombuffer(raw, dt, cnt, pos).reshape((int(m), int(n)), order="F"))
        pos += cnt * np.dtype(dt).itemsize
    return outs


@pytest.mark.parametrize("binary", [False, True])
def test_mex_globalsets_verb_matches_the_global_verb(aps, tmp_path, binary):
    sets = _mixed_sets(aps, "orb" if binary else "sift", 32 if binary else 128)
    cls = 4 if binary else 0
    nums = [len(s) for s in sets]
    got = _run_gate([(cls, m) for s in sets for m in s], [2, len(sets)] + nums + [4, 0.8, int(binary)], tmp_path)
    pos, nrows = 0, 0
    for s in sets:
        n = len(s)
        ncell = n * (n - 1) // 2
        if all(m.shape[0] == 0 for m in s):   # 'global' returns cell(numImg) without a call
            exp = [None] * ncell
        else:
            exp = _run_gate([(cls, m) for m in s], [0, 4, 0.8, int(binary)], tmp_path)
        for g, e in zip(got[pos:pos + ncell], exp):
            assert (g is None) == (e is None)
            if g is not None:
                assert g.shape == e.shape and np.array_equal(g, e)
                nrows += g.shape[0]
        pos += ncell
    assert pos == len(got) and nrows > 100
