"""Generates tests/golden/eval_metrics.npz from the reference's OWN compiled implicit/evaluation.pyx
(oracle/_ref/evaluation*.so).  Run where /root/reference exists:

    python tests/golden/make_golden_eval.py

The "model" is a table of precomputed ranked ids, so the fixture pins the metric arithmetic alone:
inputs (ids table, train/test CSR) are rebuilt from the seeds recorded in the file.

eval_ref.npz (written alone with --ref-checks) holds the reference's side of the other comparisons in
tests/test_evaluation.py: the metrics of the same cases at a second cutoff, and leave_k_out_split's held-out counts.
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

import oracle  # noqa: E402
from helpers import LEAVE_K_OUT_K, eval_case, eval_second_cutoff, leave_k_out_ratings  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = {"a": dict(users=2500, items=400, K=10, seed=31), "b": dict(users=300, items=60, K=25, seed=32),
         "c": dict(users=50, items=12, K=3, seed=33)}


def main():
    ev = oracle.ref_evaluation()
    out = {}
    for name, rc in CASES.items():
        model, train, test = eval_case(**rc)
        m = ev.ranking_metrics_at_k(model, train, test, K=rc["K"], show_progress=False)
        print(name, m)
        for k, v in m.items():
            out[f"{name}_{k}"] = np.float64(v)
        for k, v in rc.items():
            out[f"{name}_recipe_{k}"] = np.asarray(v)
        tr, te = ev.train_test_split(train + test, 0.7, rc["seed"])
        out[f"{name}_split_train_nnz"] = np.int64(tr.nnz)
        out[f"{name}_split_test_indices"] = te.indices.astype(np.int32)
    np.savez_compressed(os.path.join(HERE, "eval_metrics.npz"), **out)
    ref_checks()


def ref_checks():
    ev = oracle.ref_evaluation()
    out = {}
    for name, rc in CASES.items():
        model, train, test = eval_case(**rc)
        m = ev.ranking_metrics_at_k(model, train, test, K=eval_second_cutoff(rc["K"]), show_progress=False)
        for k, v in m.items():
            out[f"{name}_{k}"] = np.float64(v)
    mat = leave_k_out_ratings()
    for K in LEAVE_K_OUT_K:
        train, test = ev.leave_k_out_split(mat, K=K, random_state=1)
        assert ((train + test) - mat).nnz == 0
        out[f"leave_k_out_held_K{K}"] = np.diff(test.indptr).astype(np.int32)
    print(out)
    np.savez_compressed(os.path.join(HERE, "eval_ref.npz"), **out)


if __name__ == "__main__":
    ref_checks() if "--ref-checks" in sys.argv else main()
