"""featureMatchingPairwise over many independent image sets in one call (aps_feature_matching_pairwise_sets): every
set's lists (cells and metric) are bit-identical to featureMatchingPairwise on that set alone, for every method and for
binary descriptors, and to the oracle where that is cheap; a 'subsetpdist2' subset is keyed by the image's index in
its own set; sets never see each other; the pooled pass's launch count does not grow with the number of sets."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

THR, RATIO = 1.5, 0.75


@pytest.fixture(scope="module")
def ctx(aps):
    return aps._lib.default_context()


def _inp(method="exhaustive", **kw):
    d = {"Matchingmethod": "Exhaustive", "Matchingthreshold": THR, "Ratiothreshold": RATIO, "useMATLABFeatureMatch": 0}
    if method != "exhaustive":
        d.update(Matchingmethod="Approximate", ApproxFloatNNMethod=method)
    d.update(kw)
    return d


def _same(got, exp, n):
    """bit for bit: cell sizes (pair_ptr), rows and metric; returns the number of match rows"""
    (gm, gd), (em, ed) = got, exp
    rows = 0
    assert len(gm) == n and len(em) == n
    for i in range(n):
        for j in range(n):
            g, e = np.asarray(gm[i][j]), np.asarray(em[i][j])
            assert g.shape == e.shape and g.dtype == e.dtype and np.array_equal(g, e), (i, j, g.shape, e.shape)
            assert (gd[i][j] is None) == (ed[i][j] is None), (i, j)
            if gd[i][j] is not None:
                assert np.array_equal(gd[i][j], ed[i][j]), (i, j)
            rows += g.shape[0] if g.ndim == 2 else 0
    return rows


def _check(aps, sets, inp, ctx):
    """the sets call against featureMatchingPairwise per set; returns (lists, total match rows)"""
    nums = [len(s) for s in sets]
    got = aps.featureMatchingPairwiseSets(inp, sets, nums, ctx=ctx, return_metric=True)
    assert len(got) == len(sets)
    rows = 0
    for b, s in enumerate(sets):
        rows += _same(got[b], aps.featureMatchingPairwise(inp, s, nums[b], ctx=ctx, return_metric=True), nums[b])
    return got, rows


def _kaze(aps, counts, seed, scale=(), kind="kaze", D=64):
    """len(counts) ring-overlapping images cut to counts[i] rows; images listed in `scale` get max|x| > 2"""
    imgs = aps.synth.synth_descriptors(kind, len(counts), max(300, max(counts)), D, seed)
    out = [np.ascontiguousarray(im[:c]) for im, c in zip(imgs, counts)]
    for i in scale:
        out[i] = out[i] * np.float32(4.0)
    return out


# set shapes (rows per image; '*' = scaled past max|x| = 2): a mixed set (both views, mixed pairs), one image, an
# all-empty set, empty images inside a set, tiny images, two scaled images, an unscaled pair
SHAPES = [([300, 250, 173], (1,)), ([300], ()), ([0, 0], ()), ([200, 0, 150, 99], (0, 2)), ([2, 1], ()),
          ([280, 260], (0, 1)), ([300, 300], ())]


def _mixed_sets(aps, kind="kaze", D=64):
    return [_kaze(aps, sh, 700 + b, sc if kind != "orb" else (), kind, D) for b, (sh, sc) in enumerate(SHAPES)]


@pytest.mark.parametrize("method", ["exhaustive", "kdtree", "pca2nn", "subsetpdist2"])
def test_float_sets_match_single_set_calls(aps, orc, ctx, method):
    sets = _mixed_sets(aps)
    got, rows = _check(aps, sets, _inp(method), ctx)
    assert rows > 200
    for b, s in enumerate(sets):   # the oracle's restatement of each pair
        n = len(s)
        for j in range(n):
            for i in range(j):
                if s[i].shape[0] == 0 or s[j].shape[0] == 0:
                    continue
                if method == "exhaustive":
                    m, d = orc.match_features(s[i], s[j], THR, RATIO)
                elif method == "pca2nn":
                    m, d = orc.match_features_pca(s[i], s[j], THR, RATIO)
                else:
                    m, d = orc.match_features_method(s[i], s[j], THR, RATIO, method)
                assert np.array_equal(got[b][0][i][j], m.astype(np.float64)), (b, i, j)
                assert len(m) == 0 or np.array_equal(got[b][1][i][j], d), (b, i, j)


def test_float_sets_against_the_oracle_pairwise_restatement(aps, orc, ctx):
    sets = _mixed_sets(aps)
    got = aps.featureMatchingPairwiseSets(_inp(), sets, [len(s) for s in sets], ctx=ctx)
    for b, s in enumerate(sets):
        ref = orc.feature_matching_pairwise(s, THR, RATIO)["cells"]
        for j in range(len(s)):
            for i in range(j):
                e = ref.get((i, j))
                assert (e is None and got[b][i][j].shape[0] == 0) or np.array_equal(got[b][i][j], e), (b, i, j)


def test_subsetpdist2_keys_each_subset_by_the_set_local_index(aps, orc, ctx):
    """images above the subset size in different sets at different pooled positions: each set's lists equal its
    single-set plan's, whose subset tables the oracle restates (a key from the pooled index would draw other rows)"""
    subset = 500
    shapes = [[900, 300, 700], [300, 800, 650, 200], [100], [760, 540]]
    sets = [_kaze(aps, sh, 40 + b) for b, sh in enumerate(shapes)]
    inp = _inp("subsetpdist2", apsSubset=subset, apsSeed=7)
    got, rows = _check(aps, sets, inp, ctx)
    assert rows > 200
    nbig = 0
    for b, s in enumerate(sets):
        plan = aps.PairwisePlan(ctx, [d.shape[0] for d in s], 64, False)
        plan.set_method("subsetpdist2", subset=subset, seed=7)
        plan.upload(s)
        plan.prepare()
        tables = {j: plan.subset_table(j) for j, d in enumerate(s) if d.shape[0] > subset}
        plan.close()
        nbig += len(tables)
        for j in range(len(s)):
            for i in range(j):
                if j in tables:
                    m, d = orc.match_features_subset(s[i], s[j], tables[j], THR, RATIO)
                else:
                    m, d = orc.match_features_method(s[i], s[j], THR, RATIO, "subsetpdist2")
                assert np.array_equal(got[b][0][i][j], m.astype(np.float64)), (b, i, j)
                assert len(m) == 0 or np.array_equal(got[b][1][i][j], d), (b, i, j)
    assert nbig == 6   # two images above the subset size in each of sets 0, 1 and 3


@pytest.mark.parametrize("method", ["exhaustive", "subsetpdist2"])
def test_binary_sets_match_single_set_calls(aps, orc, ctx, method):
    sets = [[aps.binaryFeatures(m) for m in s] for s in _mixed_sets(aps, "orb", 32)]
    inp = _inp(method, Matchingthreshold=40.0)
    got, rows = _check(aps, sets, inp, ctx)
    assert rows > 100
    raw = _mixed_sets(aps, "orb", 32)[0]
    for j in range(3):
        for i in range(j):
            m, _ = orc.match_features(raw[i], raw[j], 40.0, RATIO)
            assert np.array_equal(got[0][0][i][j], m.astype(np.float64))


@pytest.mark.parametrize("engine", [0, 1])
def test_tensor_sized_and_tiny_sets_in_one_call(aps, ctx, engine):
    """sets the single-set call runs on the tensor path (screen + tcgen05) next to tiny exact-engine sets"""
    big = [_kaze(aps, [2048, 2100, 2048], 1700, (1,)), _kaze(aps, [2300, 0, 2048, 1900], 1701)]
    tiny = _mixed_sets(aps)[:3]
    sets = [big[0], tiny[0], big[1], tiny[1], tiny[2]]
    ctx.set_float_engine(engine)
    try:
        _, rows = _check(aps, sets, _inp(), ctx)
        aps.featureMatchingPairwiseSets(_inp(), sets, [len(s) for s in sets], ctx=ctx)
        st, ps = ctx.last_stats(), ctx.pairwise_stats()
    finally:
        ctx.set_float_engine(0)
    assert rows > 2000 and st["rows"] > 0
    if engine == 0:   # the two tensor-sized sets' 3 + 3 pairs are screened, the tiny sets' pairs are not
        assert st["engine"] == "tcgen05" and ps["pairs_screened"] == 3 + 3
    else:
        assert st["engine"] == "exact" and ps["pairs_screened"] == 0


def test_sets_are_isolated(aps, ctx):
    """set 1 holds exact copies of set 0's images; replacing set 2's descriptors changes no other set's lists"""
    a = _kaze(aps, [300, 280, 260], 11, (2,))
    b = [a[0].copy(), a[1][:200].copy()] + _kaze(aps, [240], 12)
    c = _kaze(aps, [250, 250, 250], 13)
    got, _ = _check(aps, [a, b, c], _inp(), ctx)
    c2 = _kaze(aps, [250, 250, 250], 14)
    got2, _ = _check(aps, [a, b, c2], _inp(), ctx)
    for s in (0, 1):
        _same(got2[s], got[s], len([a, b][s]))


def test_column_major_input(aps, ctx):
    sets = [[np.asfortranarray(m) for m in s] for s in _mixed_sets(aps)]
    _check(aps, sets, _inp(), ctx)
    _check(aps, [[aps.binaryFeatures(np.asfortranarray(m)) for m in s] for s in _mixed_sets(aps, "orb", 32)],
           _inp(Matchingthreshold=40.0), ctx)


def test_one_set_call_is_the_single_set_call(aps, ctx):
    desc, _ = aps.synth.make_config(5, n=30, kp=1024)   # one C5 ring
    got = aps.featureMatchingPairwiseSets(_inp(), [desc], [30], ctx=ctx, return_metric=True)
    assert _same(got[0], aps.featureMatchingPairwise(_inp(), desc, 30, ctx=ctx, return_metric=True), 30) > 1000


@pytest.mark.parametrize("shape, method", [([150, 130, 120], "exhaustive"), ([2048, 2048, 2048], "exhaustive"),
                                           ([900, 700, 300], "subsetpdist2")], ids=["small", "tensor", "subset"])
def test_launch_count_does_not_grow_with_the_number_of_sets(aps, ctx, shape, method):
    L = aps._lib.lib()
    inp = _inp(method, apsSubset=500)
    base = _kaze(aps, shape, 8000)
    delta = {}
    for B in (2, 200):
        sets = [[m[np.random.default_rng(b).permutation(m.shape[0])] for m in base] for b in range(B)]
        aps.featureMatchingPairwiseSets(inp, sets, [len(shape)] * B, ctx=ctx)   # warm-up
        n0 = L.aps_launch_count()
        aps.featureMatchingPairwiseSets(inp, sets, [len(shape)] * B, ctx=ctx)
        delta[B] = L.aps_launch_count() - n0
    assert 0 < delta[200] <= delta[2], delta


# ---- the MEX verb through the shim driver, against the per-set 'pairwise' verb -----------------------------------
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
def test_mex_pairwisesets_verb_matches_the_pairwise_verb(aps, tmp_path, binary):
    sets = _mixed_sets(aps, "orb", 32) if binary else _mixed_sets(aps)
    cls = 4 if binary else 0
    thr, method = (40.0, 0) if binary else (THR, 1)
    nums = [len(s) for s in sets]
    got = _run_gate([(cls, m) for s in sets for m in s], [3, len(sets)] + nums + [thr, RATIO, method], tmp_path)
    pos, nrows = 0, 0
    for s in sets:
        n = len(s)
        ncell = n * (n - 1) // 2
        if all(m.shape[0] == 0 for m in s):   # 'pairwise' returns cell(numImg) without a call
            exp = [None] * ncell
        else:
            exp = _run_gate([(cls, m) for m in s], [1, thr, RATIO, method], tmp_path)
        for g, e in zip(got[pos:pos + ncell], exp):
            assert (g is None) == (e is None)
            if g is not None:
                assert g.shape == e.shape and np.array_equal(g, e)
                nrows += g.shape[0]
        pos += ncell
    assert pos == len(got) and nrows > 100
