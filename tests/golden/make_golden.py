"""Generates tests/golden/*.npz from the reference's OWN compiled code (oracle/_ref, built by
oracle/build_ref.py from /root/reference).  Run where /root/reference exists:

    OPENBLAS_NUM_THREADS=1 python tests/golden/make_golden.py

Inputs are NOT stored: every case is rebuilt from implicit_b200.synthetic with the seed recorded in
the file, so a fixture is (recipe, expected outputs of the reference).  Outputs are float32.

port_vs_ref.npz (written alone with --port-vs-ref) holds the reference's side of tests/test_oracle.py's port-vs-
reference checks; their warm states are reference outputs too, so they are stored, for a sample of the rows.
"""
import os
import sys

os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import oracle  # noqa: E402
from helpers import REF_ROWS, TIES_K, WIDE_ROWS, ref_half_case, ref_wide_case, ties_case  # noqa: E402
from implicit_b200 import synthetic  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))

#: name -> recipe
CASES = {
    "chol_f16": dict(users=400, items=250, nnz=4000, factors=16, use_cg=False, iterations=2, seed=11, neg=0.0),
    "chol_f64": dict(users=300, items=200, nnz=6000, factors=64, use_cg=False, iterations=2, seed=12, neg=0.0),
    "chol_f64_neg": dict(users=300, items=200, nnz=6000, factors=64, use_cg=False, iterations=1, seed=13, neg=0.1),
    "chol_f40": dict(users=200, items=150, nnz=3000, factors=40, use_cg=False, iterations=1, seed=14, neg=0.0),
    "cg_f32": dict(users=400, items=250, nnz=5000, factors=32, use_cg=True, iterations=3, seed=15, neg=0.0),
    "cg_f128": dict(users=250, items=200, nnz=25000, factors=128, use_cg=True, iterations=3, seed=16, neg=0.05),
}


def build_case(rc):
    Cui = synthetic.power_law_csr(rc["users"], rc["items"], rc["nnz"], rc["seed"], rc["neg"])
    X0, Y0 = synthetic.initial_factors(rc["users"], rc["items"], rc["factors"], seed=42)
    return Cui, X0, Y0


def main():
    ref = oracle.get("ref")
    for name, rc in CASES.items():
        Cui, X, Y = build_case(rc)
        oracle.fit(Cui, X, Y, regularization=0.01, iterations=rc["iterations"], use_cg=rc["use_cg"], kind="ref")
        loss = ref.calculate_loss(Cui, X, Y, 0.01)
        # one more USER half from this (well conditioned) state: the tight per-half parity fixture.
        # X, Y above double as its inputs; Xh is the expected output.
        Xh = X.copy()
        if rc["use_cg"]:
            ref.least_squares_cg(Cui, Xh, Y, 0.01, cg_steps=3)
        else:
            ref.least_squares(Cui, Xh, Y, 0.01)
        ids, scores = ref.topk(Y, X[:64], 10, filter_query_items=Cui[:64], filter_items=np.array([0, 3, 7]))
        np.savez_compressed(os.path.join(HERE, name + ".npz"), X=X, Y=Y, Xh=Xh, loss=np.float64(loss), topk_ids=ids,
                            topk_scores=scores, **{"recipe_" + k: np.asarray(v) for k, v in rc.items()})
        print(name, "loss", loss, X.shape, Y.shape)
    port_vs_ref()


def port_vs_ref():
    """tests/golden/port_vs_ref.npz: what tests/test_oracle.py compares the C restatement with."""
    ref = oracle.get("ref")
    out = {}
    n = REF_ROWS
    for name, use_cg in (("chol", False), ("cg", True)):
        # one half from the reference's own warm state (two iterations)
        Cui, X, Y = ref_half_case()
        oracle.fit(Cui, X, Y, iterations=2, use_cg=use_cg, kind="ref")
        Xh = X.copy()
        if use_cg:
            ref.least_squares_cg(Cui, Xh, Y, 0.01, cg_steps=3)
        else:
            ref.least_squares(Cui, Xh, Y, 0.01)
        out.update({f"{name}_Y": Y, f"{name}_X": X[:n], f"{name}_Xh": Xh[:n],
                    f"{name}_loss": np.float64(ref.calculate_loss(Cui[:n], Xh[:n], Y, 0.01))})
    Cui, X, Y = ref_wide_case()
    n = WIDE_ROWS
    ref.least_squares_cg(Cui, X, Y, 0.01, cg_steps=3)
    ids, scores = ref.topk(Y, X[:20], 7, filter_query_items=Cui[:20])
    out.update(wide_Xh=X[:n], wide_loss=np.float64(ref.calculate_loss(Cui[:n], X[:n], Y, 0.01)), wide_topk_ids=ids,
               wide_topk_scores=scores)
    items, q = ties_case()
    for k in TIES_K:
        out[f"ties_ids_k{k}"], out[f"ties_scores_k{k}"] = ref.topk(items, q, k)
    np.savez_compressed(os.path.join(HERE, "port_vs_ref.npz"), **out)
    print("port_vs_ref", sorted(out))


if __name__ == "__main__":
    port_vs_ref() if "--port-vs-ref" in sys.argv else main()
