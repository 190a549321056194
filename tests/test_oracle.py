"""CPU-only: pins the oracle (oracle/als_oracle.c) against
  (1) the golden vectors generated from the reference's own compiled Cython (tests/golden/),
  (2) that compiled reference's answers on the same inputs (tests/golden/port_vs_ref.npz),
  (3) the known-answer / property tests the reference holds for this path."""
import os

import numpy as np
import pytest
from scipy.sparse import csr_matrix

import oracle
from helpers import (CHOL_MAX, GOLDEN, REF_ROWS, TIES_K, WIDE_ROWS, golden_cases, load_golden, ref_half_case,
                     ref_wide_case, row_err, ties_case)

PORT = oracle.get("port")
REF = np.load(os.path.join(GOLDEN, "port_vs_ref.npz"))


@pytest.mark.parametrize("name", golden_cases())
def test_port_matches_golden_warm_half(name):
    """One half-iteration from the stored (well conditioned) state: the tight per-half parity bar."""
    rc, Cui, _, _, z = load_golden(name)
    Xh = z["X"].copy()
    if rc["use_cg"]:
        PORT.least_squares_cg(Cui, Xh, z["Y"], 0.01, cg_steps=3)
    else:
        PORT.least_squares(Cui, Xh, z["Y"], 0.01)
    assert row_err(Xh, z["Xh"]).max() < 1e-5


@pytest.mark.parametrize("name", golden_cases())
def test_port_matches_golden_fit(name):
    rc, Cui, X, Y, z = load_golden(name)
    oracle.fit(Cui, X, Y, regularization=0.01, iterations=rc["iterations"], use_cg=rc["use_cg"], kind="port")
    e = np.concatenate([row_err(X, z["X"]), row_err(Y, z["Y"])])
    loss = PORT.calculate_loss(Cui, X, Y, 0.01)
    if rc["use_cg"]:
        # truncated CG from the near rank-1 random start is chaotic in factor space (SURVEY.md 8(c)):
        # two correct fp32 executions agree in loss, not row by row
        assert abs(loss - float(z["loss"])) / float(z["loss"]) < 2e-3
        assert np.median(e) < 1e-2
    else:
        assert e.max() < CHOL_MAX
        assert abs(loss - float(z["loss"])) / float(z["loss"]) < 1e-5


@pytest.mark.parametrize("name", golden_cases())
def test_port_loss_and_topk_match_golden(name):
    rc, Cui, _, _, z = load_golden(name)
    loss = PORT.calculate_loss(Cui, z["X"], z["Y"], 0.01)
    assert loss == pytest.approx(float(z["loss"]), rel=1e-6)
    ids, scores = PORT.topk(z["Y"], z["X"][:64], 10, filter_query_items=Cui[:64], filter_items=np.array([0, 3, 7]))
    np.testing.assert_allclose(scores, z["topk_scores"], rtol=1e-5, atol=1e-7)
    # ids may differ only where the reference's own scores tie to within rounding
    diff = ids != z["topk_ids"]
    if diff.any():
        assert np.abs(scores[diff] - z["topk_scores"][diff]).max() < 1e-6


@pytest.mark.parametrize("use_cg", [False, True])
def test_port_matches_compiled_reference(use_cg):
    """One half from the reference's warm state (two reference iterations), against the reference's half."""
    name = "cg" if use_cg else "chol"
    Cui = ref_half_case()[0][:REF_ROWS]
    Yw, Xa = REF[f"{name}_Y"], REF[f"{name}_Xh"]
    Xb = REF[f"{name}_X"].copy()
    if use_cg:
        PORT.least_squares_cg(Cui, Xb, Yw, 0.01, cg_steps=3)
    else:
        PORT.least_squares(Cui, Xb, Yw, 0.01)
    assert row_err(Xb, Xa).max() < 1e-5
    assert PORT.calculate_loss(Cui, Xa, Yw, 0.01) == pytest.approx(float(REF[f"{name}_loss"]), rel=1e-6)


def test_port_matches_compiled_reference_on_a_wide_model():
    """192 factors (the widths of tests/test_gpu_wide.py): the checker itself must not care about the width."""
    Cui, X, Y = ref_wide_case()
    Cui, Xa = Cui[:WIDE_ROWS], REF["wide_Xh"]
    Xb = X[:WIDE_ROWS].copy()
    PORT.least_squares_cg(Cui, Xb, Y, 0.01, cg_steps=3)
    assert row_err(Xb, Xa).max() < 1e-5
    assert PORT.calculate_loss(Cui, Xa, Y, 0.01) == pytest.approx(float(REF["wide_loss"]), rel=1e-6)
    ib, sb = PORT.topk(Y, Xa[:20], 7, filter_query_items=Cui[:20])
    np.testing.assert_allclose(sb, REF["wide_topk_scores"], rtol=1e-5, atol=1e-7)
    assert (REF["wide_topk_ids"] == ib).mean() > 0.98


# ---- the reference's own known-answer tests for this path ------------------------------------------
@pytest.mark.parametrize("use_cg", [False, True])
def test_factorize(use_cg):
    """tests/als_test.py:142-186: X Y^T must reconstruct a 7x6 binary matrix to 1e-3."""
    counts = csr_matrix(
        [[1, 1, 0, 1, 0, 0], [0, 1, 1, 1, 0, 0], [1, 0, 1, 0, 0, 0], [1, 1, 0, 0, 0, 0], [0, 0, 1, 1, 0, 1],
         [0, 1, 0, 0, 0, 1], [0, 0, 0, 0, 1, 1]], dtype=np.float64)
    rng = np.random.default_rng(23)
    X = (rng.random((7, 6), dtype=np.float32) * 0.01).astype(np.float32)
    Y = (rng.random((6, 6), dtype=np.float32) * 0.01).astype(np.float32)
    oracle.fit(counts, X, Y, regularization=0, iterations=15, use_cg=use_cg, alpha=2.0, kind="port")
    rec = X.dot(Y.T)
    dense = counts.toarray()
    for r in range(7):
        for c in range(6):
            assert dense[r, c] == pytest.approx(rec[r, c], abs=1e-3)


def test_calculate_loss_simple():
    """tests/als_test.py:304-324: the only user liked item 0; factors are perfectly wrong -> loss 1.0 (lambda=0),
    2.0 (lambda=1)."""
    from scipy.sparse import coo_matrix

    ratings = coo_matrix(([1.0], ([0], [0])), shape=(1, 2)).tocsr()
    item_factors = np.array([[0.0], [1.0]], dtype="float32")
    user_factors = np.array([[1.0]], dtype="float32")
    assert PORT.calculate_loss(ratings, user_factors, item_factors, 0) == pytest.approx(1.0)
    assert PORT.calculate_loss(ratings, user_factors, item_factors, 1.0) == pytest.approx(2.0)


def test_empty_rows_are_zeroed():
    """_als.pyx:98-100 / :182-184"""
    Cui = csr_matrix(np.array([[0, 0, 0], [1, 0, 2], [0, 0, 0]], dtype=np.float32))
    Y = np.random.default_rng(0).random((3, 8), dtype=np.float32)
    for cg in (False, True):
        X = np.ones((3, 8), dtype=np.float32)
        (PORT.least_squares_cg if cg else PORT.least_squares)(Cui, X, Y, 0.1)
        assert np.all(X[0] == 0) and np.all(X[2] == 0) and np.any(X[1] != 0)


def test_cholesky_failure_raises():
    """_als.pyx:131-138: singular normal equations with no regularization raise ValueError."""
    Cui = csr_matrix(np.array([[1.0, 0.0]], dtype=np.float32))
    Y = np.zeros((2, 4), dtype=np.float32)
    X = np.zeros((1, 4), dtype=np.float32)
    with pytest.raises(ValueError):
        PORT.least_squares(Cui, X, Y, 0.0)


def test_select_tie_semantics():
    """implicit/cpu/select.h:12-39: strict `>` admission, evict the lexicographic (score, col) minimum,
    output descending by (score, col); rows shorter than k keep their zero tail (topk.pyx:20-21)."""
    items = np.array([[5.0], [5.0], [7.0]], dtype=np.float32)
    ids, sc = PORT.topk(items, np.array([[1.0]], dtype=np.float32), 2)
    assert ids.tolist() == [[2, 1]] and sc.tolist() == [[7.0, 5.0]]
    items = np.array([[7.0], [5.0], [5.0]], dtype=np.float32)
    ids, sc = PORT.topk(items, np.array([[1.0]], dtype=np.float32), 2)
    assert ids.tolist() == [[0, 1]]
    items = np.array([[1.0], [1.0], [1.0], [1.0]], dtype=np.float32)
    ids, _ = PORT.topk(items, np.array([[1.0]], dtype=np.float32), 3)
    assert ids.tolist() == [[2, 1, 0]]
    ids, sc = PORT.topk(items[:2], np.array([[1.0]], dtype=np.float32), 4)
    assert ids.tolist() == [[1, 0, 0, 0]] and sc.tolist() == [[1.0, 1.0, 0.0, 0.0]]


def test_select_matches_compiled_reference_on_ties():
    items, q = ties_case()
    for k in TIES_K:
        b = PORT.topk(items, q, k)
        np.testing.assert_array_equal(REF[f"ties_ids_k{k}"], b[0])
        np.testing.assert_array_equal(REF[f"ties_scores_k{k}"], b[1])
