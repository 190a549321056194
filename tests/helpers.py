"""Shared helpers for the test-suite: parity metric and golden-case reconstruction."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from implicit_b200 import synthetic  # noqa: E402

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

#: Parity bars (north_star: rtol=1e-4 fp32 per factor row).  Row error = ||a - b||_2 / max(||b||_2, 1% of the
#: median row norm): elementwise rtol is unsatisfiable even by the reference against itself (SURVEY.md 8(c)).
CHOL_MAX = 1e-4
#: Truncated CG(3) amplifies rounding: the reference's own fp32 vs fp64 runs differ by up to 7e-4 on
#: iteration 1 (SURVEY.md 8(c)), so a half-iteration is gated on median / p99 and max only on a
#: converged fit.
CG_MEDIAN = 5e-5
CG_P99 = 1e-3
CG_CONVERGED_MAX = 1e-4


def row_err(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    num = np.linalg.norm(a - b, axis=1)
    den = np.linalg.norm(b, axis=1)
    floor = 0.01 * np.median(den) if len(den) else 0.0
    return num / np.maximum(np.maximum(den, floor), 1e-30)


def golden_cases():
    """The fit fixtures (chol_*, cg_*); eval_metrics.npz belongs to tests/test_evaluation.py."""
    return sorted(f[:-4] for f in os.listdir(GOLDEN) if f.endswith(".npz") and f.startswith(("chol_", "cg_")))


def load_golden(name):
    """Returns (recipe dict, Cui, X0, Y0, expected npz dict)."""
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    rc = {k[len("recipe_"):]: z[k].item() for k in z.files if k.startswith("recipe_")}
    Cui = synthetic.power_law_csr(rc["users"], rc["items"], rc["nnz"], rc["seed"], rc["neg"])
    X0, Y0 = synthetic.initial_factors(rc["users"], rc["items"], rc["factors"], seed=42)
    return rc, Cui, X0, Y0, z


# ----------------------------------------------------------------------------- port-vs-reference fixtures
#: tests/golden/port_vs_ref.npz keeps the factor rows of the first REF_ROWS / WIDE_ROWS users only: rows solve
#: independently, and power_law_csr permutes the users, so the first rows are a random sample of the matrix.
REF_ROWS = 100
WIDE_ROWS = 48
TIES_K = (1, 5, 32, 250)


def ref_half_case():
    """500 x 300, 6000 nnz with 5 % negative weights, 48 factors, from the initial factors."""
    Cui = synthetic.power_law_csr(500, 300, 6000, 77, negative_fraction=0.05)
    X0, Y0 = synthetic.initial_factors(500, 300, 48)
    return Cui, X0, Y0


def ref_wide_case():
    """192 factors (the widths of tests/test_gpu_wide.py) from random factors."""
    Cui = synthetic.power_law_csr(200, 150, 3000, 78, negative_fraction=0.05)
    rng = np.random.default_rng(5)
    X = (rng.standard_normal((200, 192)) * 0.1).astype(np.float32)
    Y = (rng.standard_normal((150, 192)) * 0.1).astype(np.float32)
    return Cui, X, Y


def ties_case():
    """Small-integer items and queries: many exact score ties."""
    rng = np.random.default_rng(5)
    items = rng.integers(0, 4, size=(200, 3)).astype(np.float32)
    q = rng.integers(0, 3, size=(17, 3)).astype(np.float32)
    return items, q


# ----------------------------------------------------------------------------- evaluation fixtures
class TableModel:
    """Stands in for a fitted model: `recommend` returns precomputed ranked ids (no GPU involved)."""

    def __init__(self, table):
        self.table = table

    def recommend(self, userid, user_items, N=10, **kwargs):
        ids = self.table[np.asarray(userid)][:, :N]
        return ids, np.zeros(ids.shape, dtype=np.float32)


def eval_case(users, items, K, seed):
    """Seeded (model, train, test): a random ranking per user, a test CSR with duplicates and empty rows."""
    import scipy.sparse as sp

    rng = np.random.default_rng(seed)
    table = np.argsort(rng.random((users, items)), axis=1)[:, :max(K, 1)].astype(np.int32)
    n = rng.integers(0, min(items, 2 * K) + 1, size=users)
    n[rng.random(users) < 0.2] = 0  # users without withheld items are skipped (evaluation.pyx:421-422)
    indptr = np.concatenate([[0], np.cumsum(n)]).astype(np.int32)
    indices = rng.integers(0, items, size=int(indptr[-1])).astype(np.int32)  # duplicates on purpose
    test = sp.csr_matrix((np.ones(len(indices), dtype=np.float32), indices, indptr), shape=(users, items))
    train = sp.random(users, items, density=0.05, format="csr", dtype=np.float32, random_state=seed)
    return TableModel(table), train, test


def eval_second_cutoff(K):
    """The cutoff tests/golden/eval_ref.npz holds the reference's metrics at, besides each case's own K."""
    return max(1, K // 2)


LEAVE_K_OUT_K = (1, 3)


def leave_k_out_ratings():
    import scipy.sparse as sp

    return sp.random(100, 100, density=0.5, format="csr", dtype=np.float32, random_state=5).tocoo()
