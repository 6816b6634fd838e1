"""CPU: the adversarial inputs of tests/test_gpu_tc_contract.py do what they are built for -- rounding directions,
approximate vs exact order, and an inflation that reaches >= 0.85 of eps_bound's operand term -- and that term is a
bound for the operand types the tensor kernels use."""
import os
import re

import numpy as np
import pytest

import tc_contract_data as tcd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_eps_terms_are_the_kernels_and_bound_the_rounding():
    src = open(os.path.join(ROOT, "automaticpanoramicimagestitching-autopanostitch-matlab_b200", "csrc",
                            "aps_exact_math.cuh")).read()
    m = re.search(r"operand_fp16 \? ([0-9.e+-]+)f : ([0-9.e+-]+)f\) \* maxsq", src)
    assert m, "eps_bound's operand term not found"
    assert float(m.group(1)) == tcd.EPS_TERM["fp16"] and float(m.group(2)) == tcd.EPS_TERM["bf16"]
    for fmt, u in tcd.UNIT_ROUNDOFF.items():
        # |a.b - a~.b~| <= (2u + u^2) sum|a_i b_i| <= (2u + u^2) max|x|^2, and the distance carries it twice
        assert 2 * (2 * u + u * u) <= tcd.EPS_TERM[fmt]


def test_unit_roundoff_matches_the_formats():
    rng = np.random.default_rng(0)
    x = (1 + rng.random(100000)).astype(np.float32)
    for fmt in ("bf16", "fp16"):
        rel = np.abs(tcd.round_operand(x, fmt).astype(np.float64) - x) / x
        u = tcd.UNIT_ROUNDOFF[fmt]
        assert rel.max() <= u and rel.max() > 0.95 * u, fmt


@pytest.mark.parametrize("fmt,kw", [("bf16", {}), ("fp16", dict(n_true=2, n_crowd=48, n_shift=40, shift_cells=4))])
def test_planted_group_rounds_against_its_true_neighbours(fmt, kw):
    rng = np.random.default_rng(5)
    g = tcd.planted_group(fmt, rng, **kw)
    n_true = kw.get("n_true", 4)
    r = tcd.round_operand(g, fmt)
    toward_zero = np.abs(r) < np.abs(g)
    assert toward_zero[:n_true].all()                    # query and true neighbours: every component
    n_up = (~toward_zero[n_true:]).sum(1)
    assert (n_up == 12).all()                           # crowd: exactly 12 components round away from zero
    q, true, crowd = g[0], g[1:n_true], g[n_true:]
    ex_true, ex_crowd = tcd.exact_l2(q, true), tcd.exact_l2(q, crowd)
    assert ex_true.max() < ex_crowd.min()               # exactly closest
    ap_true, ap_crowd = tcd.approx_l2(q, true, fmt), tcd.approx_l2(q, crowd, fmt)
    assert ap_crowd.max() < ap_true.min()               # ... but behind the whole crowd in the approximate order
    maxsq = float((g.astype(np.float64) ** 2).sum(1).max())
    term = tcd.EPS_TERM[fmt] * maxsq
    e_true = tcd.inflation(q, g[:n_true], fmt)
    e_crowd = tcd.inflation(q, crowd, fmt)
    assert e_true.max() <= term                         # the bound holds ...
    assert e_crowd.min() / term >= 0.85                 # ... with little room: a term 15 % smaller is caught
    assert e_true.max() / term >= 0.95


def test_flann_set_exact_order(orc):
    X, planted = tcd.flann_adversarial_set()
    assert X.shape == (4096, 128) and np.abs(X).max() < 16
    for qt, crowd in planted:
        oi, od = orc.knn_l2(X, X[qt[:1]], 4)
        assert set((oi[0] - 1).tolist()) == set(qt.tolist())
        assert len(crowd) >= 40


def test_pairwise_set_exact_order(orc):
    A, B, planted = tcd.pairwise_adversarial_set()
    assert np.abs(A).max() <= 2 and np.abs(B).max() <= 2   # raw fp16 operands (no normalisation)
    for ra, rb, crowd in planted:
        oi, od = orc.knn_l2(B, A[ra:ra + 1], 2)
        assert oi[0, 0] - 1 == rb and oi[0, 1] - 1 in set(crowd.tolist())
    m, met = orc.match_features(A, B, 3.5, 0.6)
    got = {(int(a) - 1, int(b) - 1) for a, b in m}
    for ra, rb, _ in planted:
        assert (ra, rb) in got                          # the planted query is a match in the reference


def test_degenerate_set():
    rng = np.random.default_rng(2)
    X = tcd.degenerate_set(20037, rng)
    assert X.shape[0] % 128 != 0
    assert ((X == 0).all(1)).sum() >= 3
    _, counts = np.unique(X, axis=0, return_counts=True)
    assert counts.max() >= 201
    assert ((X == X[:, :1]).all(1)).sum() >= 23         # constant rows (zero rows included)
