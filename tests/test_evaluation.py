"""Ranking evaluation (SURVEY.md 8(f) N4; implicit/evaluation.pyx:366-475).

CPU part: the metric arithmetic of implicit_b200.evaluation and of the oracle restatement against the
golden values produced by the reference's own compiled module (eval_metrics.npz, eval_ref.npz), with a table of
precomputed ids standing in for the model.  GPU part: the real model driving the fused top-k kernel through `recommend`."""
import os

import numpy as np
import pytest

from helpers import LEAVE_K_OUT_K, eval_case, eval_second_cutoff, leave_k_out_ratings
from oracle import evaluation_oracle

GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "eval_metrics.npz"))
REF = np.load(os.path.join(os.path.dirname(__file__), "golden", "eval_ref.npz"))
CASES = sorted({k.split("_")[0] for k in GOLD.files})
KEYS = ("precision", "map", "ndcg", "auc")


def _recipe(name):
    return {k: int(GOLD[f"{name}_recipe_{k}"]) for k in ("users", "items", "K", "seed")}


@pytest.mark.parametrize("name", CASES)
def test_oracle_restatement_matches_golden(name):
    rc = _recipe(name)
    model, train, test = eval_case(**rc)
    got = evaluation_oracle.ranking_metrics_at_k(model, train, test, K=rc["K"])
    for k in KEYS:
        assert got[k] == pytest.approx(float(GOLD[f"{name}_{k}"]), rel=1e-12)


@pytest.mark.parametrize("name", CASES)
def test_oracle_restatement_matches_compiled_reference(name):
    """The same cases at a second cutoff, below the length of the ranked lists."""
    rc = _recipe(name)
    model, train, test = eval_case(**rc)
    got = evaluation_oracle.ranking_metrics_at_k(model, train, test, K=eval_second_cutoff(rc["K"]))
    for k in KEYS:
        assert got[k] == pytest.approx(float(REF[f"{name}_{k}"]), rel=1e-12)


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("batch", [7, 16384])
def test_ranking_metrics_match_golden(name, batch, monkeypatch):
    from implicit_b200 import evaluation

    monkeypatch.setattr(evaluation, "BATCH", batch)
    rc = _recipe(name)
    model, train, test = eval_case(**rc)
    got = evaluation.ranking_metrics_at_k(model, train, test, K=rc["K"], show_progress=False)
    for k in KEYS:
        assert got[k] == pytest.approx(float(GOLD[f"{name}_{k}"]), rel=1e-12)
    assert evaluation.precision_at_k(model, train, test, K=rc["K"], show_progress=False) == got["precision"]
    assert evaluation.mean_average_precision_at_k(model, train, test, K=rc["K"], show_progress=False) == got["map"]
    assert evaluation.ndcg_at_k(model, train, test, K=rc["K"], show_progress=False) == got["ndcg"]
    assert evaluation.AUC_at_k(model, train, test, K=rc["K"], show_progress=False) == got["auc"]


@pytest.mark.parametrize("name", CASES)
def test_train_test_split_matches_golden(name):
    from implicit_b200 import evaluation

    rc = _recipe(name)
    _, train, test = eval_case(**rc)
    for impl in (evaluation, evaluation_oracle):
        tr, te = impl.train_test_split(train + test, 0.7, rc["seed"])
        assert tr.nnz == int(GOLD[f"{name}_split_train_nnz"])
        np.testing.assert_array_equal(te.indices, GOLD[f"{name}_split_test_indices"])
    tr2, _ = evaluation.train_test_split(train + test, 0.7, rc["seed"])  # tests/evaluation_test.py:22-27
    assert (tr != tr2).nnz == 0


# ---- leave_k_out_split: the reference's own property tests (tests/evaluation_test.py:30-100)
@pytest.mark.parametrize("K", LEAVE_K_OUT_K)
def test_leave_k_out_split_contract(K):
    from implicit_b200 import evaluation

    mat = leave_k_out_ratings()
    train, test = evaluation.leave_k_out_split(mat, K=K, random_state=1)
    assert train.shape == mat.shape and test.shape == mat.shape          # :30-38
    assert ((train + test) - mat).nnz == 0                                # :41-49
    assert mat.sum() > 0 and test.sum() > 0 and train.sum() > 0          # :52-66
    counts = np.bincount(mat.row, minlength=100)
    held = np.diff(test.indptr)
    assert np.all(held[counts > K + 1] == K) and np.all(held[counts <= K + 1] == 0)
    t2, _ = evaluation.leave_k_out_split(mat, K=K, random_state=1)       # seeded
    assert (t2 != train).nnz == 0
    np.testing.assert_array_equal(REF[f"leave_k_out_held_K{K}"], held)  # what the reference's compiled module holds out


def test_leave_k_out_split_train_only_and_errors():
    from implicit_b200 import evaluation

    mat = leave_k_out_ratings()
    train, test = evaluation.leave_k_out_split(mat, K=1, train_only_size=0.8, random_state=2)
    train_only = ~np.isin(np.unique(train.tocoo().row), test.tocoo().row)
    assert train_only.sum() == int(train.shape[0] * 0.8)                  # :69-76
    with pytest.raises(ValueError):
        evaluation.leave_k_out_split(None, K=0)                           # :79-84
    with pytest.raises(ValueError):
        evaluation.leave_k_out_split(None, K=1, train_only_size=-1.0)     # :87-92
    with pytest.raises(ValueError):
        evaluation.leave_k_out_split(None, K=1, train_only_size=1.0)      # :95-100


@pytest.mark.gpu
def test_evaluate_fitted_model_against_oracle_ids():
    """The model's own recommend() under ranking_metrics_at_k == the scalar restatement fed by the same
    model, and a fit on structured data scores far above chance (tests/evaluation_test.py:103-121)."""
    import scipy.sparse as sp

    from implicit_b200 import evaluation
    from implicit_b200.als import AlternatingLeastSquares

    rng = np.random.default_rng(8)
    users, items, groups = 3000, 600, 12
    ug, ig = rng.integers(0, groups, users), rng.integers(0, groups, items)
    dense = (ug[:, None] == ig[None, :]) & (rng.random((users, items)) < 0.5)
    ratings = sp.csr_matrix(dense.astype(np.float32))
    train, test = evaluation.train_test_split(ratings, 0.8, 3)
    model = AlternatingLeastSquares(factors=32, regularization=0.05, iterations=8, use_cg=False, random_state=1)
    model.fit(train, show_progress=False)
    got = evaluation.ranking_metrics_at_k(model, train, test, K=10, show_progress=False)
    exp = evaluation_oracle.ranking_metrics_at_k(model, train, test, K=10)
    for k in KEYS:
        assert got[k] == pytest.approx(exp[k], rel=1e-12)
    # likes are random WITHIN a group: of the ~30 unfiltered same-group items ~5 are withheld, so a perfect
    # group model scores 10 * (5/30) / 5 = 1/3; chance is below 0.02
    assert got["precision"] > 0.25 and got["auc"] > 0.5
