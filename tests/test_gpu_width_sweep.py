"""Every factor-width specialisation of the solvers, the loss, the Gramian and top-k against fp64 references.

The hot kernels are templates over the padded factor width `ld` (16 * ceil(f / 16) up to 128 factors, 128 * ceil(f / 128)
beyond), picked by a `switch` on ld / 16 or ld / 128:

  Cholesky   cholesky.cu run_cholesky<NB>, NB = ld / 16 = 1..4;  cholesky_wide.cu run_wide<T>, T = ld / 16 = 5..8
  CG         cg.cu run_cg<F, NV>, F = 16..128 x NV (knob cg_nv) in {1, 2, 4};  run_cg<256..1024> beyond 128
  loss       loss.cu, ld / 16 = 1..8 and ld / 128 = 2..8
  Gramian    tcgen05 + TMA (ld 64, >= 128 rows), FMA (ld 16..128), mma.sync (knob gramian_mma), wide (ld / 64)
  top-k      topk.cu run_topk_f<F> for ld <= 128, score + segmented sort beyond

Each case is compared with the CPU oracle (oracle.get("auto")) and, for the solvers and the loss, with the fp64
restatements of the reference below (chol_truth, cg_truth, loss_truth).  A GPU result must be no further from the
fp64 truth than the fp32 reference is, up to a fixed floor.  Every case prints its numbers, so a log of
`pytest -m gpu -s` records the error of every instantiation.

The tests without the `gpu` mark pin the fp64 restatements to the oracle's C port and show that every bar used here
rejects a result that is wrong by 1e-3 in one row.
"""
import contextlib

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse as sp

import oracle
from helpers import CG_MEDIAN, CG_P99, CHOL_MAX, row_err


# ======================================================================================== fp64 references
def chol_truth(Cui, Y, reg):
    """implicit/cpu/_als.pyx:76-142 in fp64, one solve per row.  A = Y^T Y + reg I + sum (|c| - 1) y y^T and
    b = sum_{c > 0} c y over the stored entries as they are: duplicates are not merged and a stored 0.0 subtracts
    y y^T.  An empty row gives zeros.  A row whose A is not positive definite raises ValueError naming the row."""
    Y64 = np.asarray(Y, dtype=np.float64)
    f = Y64.shape[1]
    G = Y64.T @ Y64 + reg * np.eye(f)
    out = np.zeros((Cui.shape[0], f))
    for u in range(Cui.shape[0]):
        s, t = Cui.indptr[u], Cui.indptr[u + 1]
        if s == t:
            continue
        Yu = Y64[Cui.indices[s:t]]
        c = Cui.data[s:t].astype(np.float64)
        A = G + (Yu.T * (np.abs(c) - 1.0)) @ Yu
        b = Yu.T @ np.where(c > 0, c, 0.0)
        try:
            out[u] = scipy.linalg.cho_solve(scipy.linalg.cho_factor(A), b)
        except np.linalg.LinAlgError:
            raise ValueError(f"cholesky failed on row {u}") from None
    return out


def cg_truth(Cui, X0, Y, reg, steps):
    """implicit/cpu/_als.pyx:154-248 in fp64: CG(steps) from X0, with both early exits (rsold < 1e-20 leaves the row
    as it was, rsnew < 1e-20 stops the iteration)."""
    Y64 = np.asarray(Y, dtype=np.float64)
    f = Y64.shape[1]
    YtY = Y64.T @ Y64 + reg * np.eye(f)
    out = np.asarray(X0, dtype=np.float64).copy()
    for u in range(Cui.shape[0]):
        s, t = Cui.indptr[u], Cui.indptr[u + 1]
        if s == t:
            out[u] = 0.0
            continue
        Yu = Y64[Cui.indices[s:t]]
        c = Cui.data[s:t].astype(np.float64)
        w = np.abs(c) - 1.0
        x = out[u]
        r = -YtY @ x + Yu.T @ (np.where(c > 0, c, 0.0) - w * (Yu @ x))
        p = r.copy()
        rsold = r @ r
        if rsold < 1e-20:
            continue
        for _ in range(steps):
            Ap = YtY @ p + Yu.T @ (w * (Yu @ p))
            alpha = rsold / (p @ Ap)
            x += alpha * p
            r -= alpha * Ap
            rsnew = r @ r
            if rsnew < 1e-20:
                break
            p = r + (rsnew / rsold) * p
            rsold = rsnew
    return out


def loss_truth(Cui, X, Y, reg):
    """implicit/cpu/_als.pyx:259-308 in fp64."""
    X64, Y64 = np.asarray(X, dtype=np.float64), np.asarray(Y, dtype=np.float64)
    rows = np.repeat(np.arange(Cui.shape[0]), np.diff(Cui.indptr))
    c = Cui.data.astype(np.float64)
    conf = np.abs(c)
    d = np.einsum("ij,ij->i", Y64[Cui.indices], X64[rows])
    t = np.where(c > 0, -2.0 * c, 0.0) + (conf - 1.0) * d
    loss = conf.sum() + np.einsum("ij,jk,ik->", X64, Y64.T @ Y64, X64) + (t * d).sum()
    loss += reg * ((Y64 ** 2).sum() + (X64 ** 2).sum())
    return loss / (conf.sum() + Cui.shape[0] * Cui.shape[1] - Cui.nnz)


# ======================================================================================== bars
#: Floors of the Cholesky bars against the fp64 truth: round-2 measurements at f = 64 (DESIGN.md sections 2, 4.1).
CHOL_TRUTH_MEDIAN = 2e-6
CHOL_TRUTH_MAX = 5e-5
#: A CG half-iteration is gated on its worst row against the oracle too, at ten times the converged-fit bar.
CG_MAX = 1e-3
LOSS_REL = 1e-5
GRAM_REL = 2e-6


def _stats(e):
    return dict(median=float(np.median(e)), p99=float(np.percentile(e, 99)), max=float(e.max()))


def chol_bars(got, exp, truth, empty):
    """{bar: passed} for a Cholesky half: `exp` is the oracle's result, `truth` chol_truth's."""
    eo, eg, er = row_err(got, exp), row_err(got, truth), row_err(exp, truth)
    return {
        "oracle max": eo.max() < CHOL_MAX,
        "truth median": np.median(eg) <= max(CHOL_TRUTH_MEDIAN, 1.5 * np.median(er)),
        "truth max": eg.max() <= max(CHOL_TRUTH_MAX, 1.5 * er.max()),
        "empty rows zero": bool(np.all(got[empty] == 0)),
    }, f"vs oracle {_fmt(eo)} | vs fp64 gpu {_fmt(eg)} oracle {_fmt(er)}"


def cg_bars(got, exp, truth, empty):
    eo, eg, er = row_err(got, exp), row_err(got, truth), row_err(exp, truth)
    return {
        "oracle median": np.median(eo) < CG_MEDIAN,
        "oracle p99": np.percentile(eo, 99) < CG_P99,
        "oracle max": eo.max() < CG_MAX,
        "truth median": np.median(eg) <= 1.5 * np.median(er),
        "truth max": eg.max() <= 1.5 * er.max(),
        "empty rows zero": bool(np.all(got[empty] == 0)),
    }, f"vs oracle {_fmt(eo)} | vs fp64 gpu {_fmt(eg)} oracle {_fmt(er)}"


def loss_bars(got, truth):
    return {"rel": abs(got - truth) <= LOSS_REL * abs(truth)}, f"loss {got:.9g} fp64 {truth:.9g} rel {abs(got - truth) / abs(truth):.2e}"


def gram_bars(G, Y):
    """|G - G64| <= 2e-6 max(|Y|^T |Y|): scaled by the sum of magnitudes, so that cancellation cannot hide an error."""
    Y64 = np.asarray(Y, dtype=np.float64)
    G64 = Y64.T @ Y64
    scale = (np.abs(Y64).T @ np.abs(Y64)).max()
    err = np.abs(G - G64).max()
    return {"scaled": err <= GRAM_REL * scale}, f"|G - G64| {err:.2e} = {err / scale:.2e} x max(|Y|^T|Y|)"


def topk_bars(ids, sc, eids, esc, query, items, filt):
    """Ids equal except at near-ties (scores within fp32 summation noise, as in test_gpu_fullsize.py); scores equal to
    rtol 1e-5 plus that noise; no filtered item returned."""
    noise = 4 * np.finfo(np.float32).eps * np.linalg.norm(query, axis=1)[:, None] * np.linalg.norm(items, axis=1).max()
    same = ids == eids
    gap = np.abs(sc.astype(np.float64) - esc)
    # the fp64 score of each returned id: where the ids differ, it must tie with the expected score at that rank
    own = np.einsum("qf,qkf->qk", np.asarray(query, np.float64), np.asarray(items, np.float64)[ids])
    return {
        "ids": not ((~same) & (np.abs(own - esc) > noise)).any(),
        "scores": bool(np.all(gap <= 1e-5 * np.abs(esc) + noise)),
        "filter": not np.isin(ids, filt).any(),
    }, f"ids equal {same.mean():.4f}, score gap max {gap.max():.2e}"


def _fmt(e):
    s = _stats(e)
    return f"med {s['median']:.1e} p99 {s['p99']:.1e} max {s['max']:.1e}"


def _check(bars, msg, label):
    print(f"{label}: {msg}")
    failed = [k for k, ok in bars.items() if not ok]
    assert not failed, f"{label}: bars {failed} missed: {msg}"


# ======================================================================================== inputs
BOUNDARY_LENGTHS = (1, 8, 9, 16, 17, 24, 32, 33, 40, 48, 49)  # the short-row size classes of cholesky_short.cu
SPLIT_NNZ = 3072  # rows longer than this take the chunk + finish path (common.h kSplitNnz)


def _row_values(rng, n, kind):
    """1..5 confidences with one kind of special entry: |c| < 1, an explicit zero, disliked (|c| >= 1), c == 1."""
    v = 1 + 4 * rng.random(n)
    if n and kind == 1:
        v[0] = 0.5
    elif n and kind == 2:
        v[0] = 0.0
    elif n and kind == 3:
        v[: n // 2 + 1] *= -1
    elif n and kind == 4:
        v[0] = 1.0
    elif n and kind == 5:
        v[0] = -0.25
    return v


def mixed_csr(seed, items, lengths, giants):
    """A CSR built from its arrays so that nothing is merged or dropped: rows of the given lengths (0 = empty), each
    with one kind of special value (see _row_values) and every 7th with a duplicated column, then the giant rows,
    which mix all kinds; the longest one draws its columns with replacement (duplicates throughout)."""
    rng = np.random.default_rng(seed)
    indices, data, indptr = [], [], [0]
    for u, n in enumerate(lengths):
        c = rng.choice(items, n, replace=False)
        if n >= 2 and u % 7 == 6:
            c[1] = c[0]
        indices.append(c)
        data.append(_row_values(rng, n, u % 7))
        indptr.append(indptr[-1] + n)
    for g, n in enumerate(giants):
        c = rng.choice(items, n, replace=n > items // 2)
        v = 1 + 4 * rng.random(n)
        v[rng.random(n) < 0.05] *= -1
        v[:4] = (0.0, 0.5, -0.25, 1.0)
        indices.append(c)
        data.append(v)
        indptr.append(indptr[-1] + n)
    Cui = sp.csr_matrix((np.concatenate(data).astype(np.float32), np.concatenate(indices).astype(np.int32),
                         np.array(indptr, dtype=np.int32)), shape=(len(lengths) + len(giants), items))
    return Cui


def chol_csr():
    """The Cholesky sweep's matrix: 20 empty rows, 60 rows at each short-class boundary length, 200 long rows of
    50..400 nonzeros and two giant rows (3100 and 8200 nonzeros) over 4000 items."""
    rng = np.random.default_rng(11)
    lengths = [0] * 20 + list(BOUNDARY_LENGTHS) * 60 + rng.integers(50, 401, 200).tolist()
    lengths = [lengths[i] for i in rng.permutation(len(lengths))]
    return mixed_csr(12, 4000, lengths, giants=(3100, 8200))


def small_csr():
    """CG, loss: 5 empty rows, 20 rows at each boundary length, 60 rows of 50..300 and giant rows of 3100 and 6500."""
    rng = np.random.default_rng(21)
    lengths = [0] * 5 + list(BOUNDARY_LENGTHS) * 20 + rng.integers(50, 301, 60).tolist()
    lengths = [lengths[i] for i in rng.permutation(len(lengths))]
    return mixed_csr(22, 7000, lengths, giants=(3100, 6500))


def factors(rows, f, seed, scale):
    return (np.random.default_rng(seed).standard_normal((rows, f)) * scale).astype(np.float32)


def padded(f):
    return 16 * -(-f // 16) if f <= 128 else 128 * -(-f // 128)


def chol_path(f):
    ld = padded(f)
    return f"NB{ld // 16}" if ld <= 64 else f"wideT{ld // 16}"


def empty_rows(Cui):
    return np.diff(Cui.indptr) == 0


# ======================================================================================== CPU: the references themselves
def _tiny_case(f, seed):
    rng = np.random.default_rng(seed)
    lengths = [0, 1, 2, 5, 9, 17, 33] * 6 + rng.integers(40, 120, 10).tolist()
    Cui = mixed_csr(seed, 300, lengths, giants=())
    X = factors(Cui.shape[0], f, seed + 1, 0.1)
    Y = factors(300, f, seed + 2, 0.2)
    return Cui, X, Y


#: Measured with oracle/als_oracle.c (gcc -O2, fp32) on these cases: Cholesky max 5e-7, CG max 2.1e-6, loss 8e-10.
PORT_CHOL_MAX, PORT_CG_MAX, PORT_LOSS_REL = 1e-5, 2e-5, 1e-7


@pytest.mark.parametrize("f", [5, 20])
def test_fp64_references_agree_with_oracle_port(f):
    """The fp64 restatements and the oracle's C port are one algorithm: they differ by fp32 rounding only."""
    Cui, X, Y = _tiny_case(f, 300 + f)
    port = oracle.get("port")
    exp = X.copy()
    port.least_squares(Cui, exp, Y, 0.05)
    e_chol = row_err(exp, chol_truth(Cui, Y, 0.05))
    exp_cg = X.copy()
    port.least_squares_cg(Cui, exp_cg, Y, 0.05, cg_steps=3)
    e_cg = row_err(exp_cg, cg_truth(Cui, X, Y, 0.05, 3))
    lt, lp = loss_truth(Cui, X, Y, 0.05), port.calculate_loss(Cui, X, Y, 0.05)
    e_loss = abs(lp - lt) / abs(lt)
    print(f"f={f}: port vs fp64: cholesky {_fmt(e_chol)}; cg {_fmt(e_cg)}; loss rel {e_loss:.1e}")
    assert e_chol.max() < PORT_CHOL_MAX and e_cg.max() < PORT_CG_MAX and e_loss < PORT_LOSS_REL
    assert np.all(exp[empty_rows(Cui)] == 0) and np.all(exp_cg[empty_rows(Cui)] == 0)
    # the fp32 port is not bit-equal to fp64 somewhere: the comparison measures something
    assert e_chol.max() > 0 and e_cg.max() > 0 and e_loss > 0


def test_fp64_cholesky_reference_raises_on_indefinite_row():
    Y = factors(50, 4, 3, 0.2)
    Cui = sp.csr_matrix((np.zeros(200, dtype=np.float32), np.full(200, 7, dtype=np.int32),
                         np.array([0, 0, 200], dtype=np.int32)), shape=(2, 50))
    with pytest.raises(ValueError, match=r"row 1\b"):
        chol_truth(Cui, Y, 0.0)
    with pytest.raises(ValueError, match=r"row 1\b"):
        oracle.get("port").least_squares(Cui, np.zeros((2, 4), dtype=np.float32), Y, 0.0)


def _perturb_row(a, row, rel=1e-3):
    b = np.array(a, dtype=np.float32, copy=True)
    d = np.random.default_rng(row).standard_normal(b.shape[1])
    b[row] += (rel * np.linalg.norm(b[row]) / np.linalg.norm(d) * d).astype(np.float32)
    return b


def test_bars_reject_one_row_off_by_1e3():
    """Every bar used on the GPU passes the oracle's own result and rejects it with one row off by 1e-3 (relative):
    the per-row max bars on that one row, the median and p99 bars when every row is off (by 2e-3: the CG p99 bar
    is 1e-3 itself).  The loss and top-k bars judge a
    scalar and a score table; one value off by 1e-3 must fail them."""
    Cui, X, Y = _tiny_case(20, 77)
    port = oracle.get("port")
    empty = empty_rows(Cui)
    row = int(np.argmax(np.diff(Cui.indptr)))
    everyone = lambda a: np.where(empty[:, None], a, a * np.float32(1 + 2e-3))  # noqa: E731

    exp = X.copy()
    port.least_squares(Cui, exp, Y, 0.05)
    truth = chol_truth(Cui, Y, 0.05)
    ok, _ = chol_bars(exp, exp, truth, empty)
    assert all(ok.values()), ok
    one, _ = chol_bars(_perturb_row(exp, row), exp, truth, empty)
    assert not one["oracle max"] and not one["truth max"], one
    allrows, _ = chol_bars(everyone(exp), exp, truth, empty)
    assert not allrows["truth median"], allrows
    assert not chol_bars(np.where(empty[:, None], 1e-30, exp), exp, truth, empty)[0]["empty rows zero"]

    exp = X.copy()
    port.least_squares_cg(Cui, exp, Y, 0.05, cg_steps=3)
    truth = cg_truth(Cui, X, Y, 0.05, 3)
    ok, _ = cg_bars(exp, exp, truth, empty)
    assert all(ok.values()), ok
    one, _ = cg_bars(_perturb_row(exp, row), exp, truth, empty)
    assert not one["truth max"], one
    allrows, _ = cg_bars(everyone(exp), exp, truth, empty)
    assert not allrows["oracle median"] and not allrows["oracle p99"] and not allrows["truth median"], allrows
    assert not cg_bars(_perturb_row(exp, row, 2e-3), exp, truth, empty)[0]["oracle max"]

    lt = loss_truth(Cui, X, Y, 0.05)
    assert loss_bars(port.calculate_loss(Cui, X, Y, 0.05), lt)[0]["rel"]
    assert not loss_bars(lt * (1 + 1e-3), lt)[0]["rel"]

    G = port.gramian(Y)
    assert gram_bars(G, Y)[0]["scaled"]
    j = int(np.argmax(np.diag(G)))
    assert not gram_bars(_perturb_row(G, j), Y)[0]["scaled"]

    items, q = factors(300, 20, 5, 0.3), factors(30, 20, 6, 0.3)
    filt = np.array([0, 7])
    ids, sc = port.topk(items, q, 10, filter_items=filt)
    assert all(topk_bars(ids, sc, ids, sc, q, items, filt)[0].values())
    assert not topk_bars(ids, _perturb_row(sc, 3), ids, sc, q, items, filt)[0]["scores"]
    swapped = ids.copy()
    swapped[3, [0, 9]] = swapped[3, [9, 0]]
    assert not topk_bars(swapped, sc, ids, sc, q, items, filt)[0]["ids"]


def test_sweep_names_every_instantiation():
    """The GPU sweep below covers every template instantiation the host code dispatches to."""
    assert sorted({chol_path(f) for f in CHOL_WIDTHS}) == sorted([f"NB{i}" for i in range(1, 5)] + [f"wideT{i}" for i in range(5, 9)])
    assert sorted({padded(f) for f in CG_NARROW}) == list(range(16, 129, 16))
    assert sorted({padded(f) for f in CG_WIDE}) == list(range(640, 1025, 128))
    assert sorted({padded(f) for f in LOSS_WIDTHS}) == list(range(16, 129, 16)) + list(range(256, 1025, 128))
    assert {padded(f) for f in GRAM_WIDTHS} >= set(range(16, 129, 16)) | set(range(640, 1025, 128))


# ======================================================================================== GPU fixtures
@pytest.fixture(scope="module")
def lib():
    from implicit_b200 import _lib

    return _lib


@pytest.fixture(scope="module")
def ctx(lib):
    c = lib.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def orc():
    return oracle.get("auto")


@pytest.fixture(scope="module")
def chol_matrix():
    return chol_csr()


@pytest.fixture(scope="module")
def small_matrix():
    return small_csr()


#: knob defaults (include/als_b200.h, common.h als_knobs)
KNOB_DEFAULTS = dict(short_max=48, short_serial=0, whiten_fma=0, gramian_mma=0, gramian_fma=0, cg_nv=2)


@contextlib.contextmanager
def knob(ctx, name, value):
    ctx.set_knob(name, value)
    try:
        yield
    finally:
        ctx.set_knob(name, KNOB_DEFAULTS[name])


class Half:
    """Device handles of one half-iteration (CSR, X, Y); closed on exit."""

    def __init__(self, lib, ctx, Cui, X, Y):
        self.lib, self.ctx = lib, ctx
        self.C = lib.DeviceCSR.upload(ctx, Cui)
        self.X = lib.DeviceFactors.from_host(ctx, X)
        self.Y = lib.DeviceFactors.from_host(ctx, Y)

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        for h in (self.C, self.X, self.Y):
            h.close()

    def chol(self, reg):
        self.lib.least_squares(self.ctx, self.C, self.X, self.Y, reg)
        return self.X.download()

    def cg(self, reg, steps=3):
        self.lib.least_squares_cg(self.ctx, self.C, self.X, self.Y, reg, steps)
        return self.X.download()


def gpu_chol(lib, ctx, Cui, Y, reg):
    with Half(lib, ctx, Cui, np.zeros((Cui.shape[0], Y.shape[1]), np.float32), Y) as h:
        return h.chol(reg)


def oracle_chol(orc, Cui, Y, reg):
    exp = np.zeros((Cui.shape[0], Y.shape[1]), dtype=np.float32)
    orc.least_squares(Cui, exp, Y, reg)
    return exp


# ======================================================================================== a. Cholesky half
CHOL_WIDTHS = [1, 8, 15, 16, 17, 31, 32, 33, 47, 48, 49, 63, 64, 65, 80, 96, 100, 112, 127, 128]
_truth_cache = {}


def _chol_case(chol_matrix, f, reg, orc):
    key = (f, reg)
    if key not in _truth_cache:
        Y = factors(chol_matrix.shape[1], f, 1000 + f, 0.2)
        _truth_cache.clear()
        _truth_cache[key] = (Y, oracle_chol(orc, chol_matrix, Y, reg), chol_truth(chol_matrix, Y, reg))
    return _truth_cache[key]


@pytest.mark.gpu
@pytest.mark.parametrize("reg", [0.01, 1.0])
@pytest.mark.parametrize("f", CHOL_WIDTHS, ids=[f"f{f}-{chol_path(f)}" for f in CHOL_WIDTHS])
def test_cholesky_half_width(lib, ctx, orc, chol_matrix, f, reg):
    Y, exp, truth = _chol_case(chol_matrix, f, reg, orc)
    got = gpu_chol(lib, ctx, chol_matrix, Y, reg)
    _check(*chol_bars(got, exp, truth, empty_rows(chol_matrix)), f"cholesky f={f} ({chol_path(f)}) reg={reg}")


@pytest.mark.gpu
@pytest.mark.parametrize("f", [17, 100], ids=["f17-NB2", "f100-wideT7"])
def test_cholesky_half_unregularised(lib, ctx, orc, chol_matrix, f):
    """reg = 0 on a well-posed case (4000 items, every row's A positive definite): the identity on the padded
    diagonal keeps the padded system solvable."""
    Y, exp, truth = _chol_case(chol_matrix, f, 0.0, orc)
    got = gpu_chol(lib, ctx, chol_matrix, Y, 0.0)
    _check(*chol_bars(got, exp, truth, empty_rows(chol_matrix)), f"cholesky f={f} reg=0")


@pytest.mark.gpu
@pytest.mark.parametrize("f", [80, 100, 112])
def test_cholesky_with_gramian_width(lib, ctx, orc, chol_matrix, f):
    """als_least_squares_with_gramian (the reference's _least_squares(YtY, ...)) on the wide kernel."""
    Y = factors(chol_matrix.shape[1], f, 2000 + f, 0.2)
    YtY = (Y.astype(np.float64).T @ Y.astype(np.float64)).astype(np.float32)
    exp = np.zeros((chol_matrix.shape[0], f), dtype=np.float32)
    orc._least_squares(YtY, chol_matrix.indptr, chol_matrix.indices, chol_matrix.data, exp, Y, 0.01)
    truth = chol_truth(chol_matrix, Y, 0.01)
    with Half(lib, ctx, chol_matrix, np.zeros_like(exp), Y) as h:
        lib.least_squares_with_gramian(ctx, YtY, h.C, h.X, h.Y, 0.01)
        got = h.X.download()
    _check(*chol_bars(got, exp, truth, empty_rows(chol_matrix)), f"with_gramian f={f}")


@pytest.mark.gpu
def test_fit_factors_100_cholesky_matches_oracle(orc):
    """factors=100 (the reference's default) through the public class: 2 iterations from injected factors."""
    from implicit_b200 import AlternatingLeastSquares, synthetic

    Cui = synthetic.power_law_csr(1500, 1000, 30000, 61, 0.05)
    X0, Y0 = factors(1500, 100, 62, 0.1), factors(1000, 100, 63, 0.1)
    Xe, Ye = X0.copy(), Y0.copy()
    oracle.fit(Cui, Xe, Ye, iterations=2, use_cg=False, kind=orc.name)
    m = AlternatingLeastSquares(factors=100, use_cg=False, iterations=2)
    m.user_factors, m.item_factors = X0.copy(), Y0.copy()
    m.fit(Cui, show_progress=False)
    e = np.concatenate([row_err(m.user_factors, Xe), row_err(m.item_factors, Ye)])
    print(f"fit factors=100 cholesky, 2 iterations: {_fmt(e)}")
    assert e.max() < CHOL_MAX


# ======================================================================================== b. not positive definite, wide kernel
def _indefinite_csr(items, bad_whole, bad_giant, rows=48, seed=0):
    """Ordinary rows of 40 nonzeros, except: `bad_whole` holds one item 600 times with c = 0.0 (plus 20 ordinary
    entries), `bad_giant` holds one item 1200 times with c = 0.0 among 3500 nonzeros (chunks + finish)."""
    rng = np.random.default_rng(seed)
    indices, data, indptr = [], [], [0]
    for u in range(rows):
        if u == bad_whole or u == bad_giant:
            reps, n = (600, 20) if u == bad_whole else (1200, 2300)
            c = np.concatenate([np.full(reps, 7 + u), rng.choice(items, n, replace=False)])
            v = np.concatenate([np.zeros(reps), 1 + 4 * rng.random(n)])
        else:
            c, v = rng.choice(items, 40, replace=False), 1 + 4 * rng.random(40)
        indices.append(c)
        data.append(v)
        indptr.append(indptr[-1] + len(c))
    return sp.csr_matrix((np.concatenate(data).astype(np.float32), np.concatenate(indices).astype(np.int32),
                          np.array(indptr, dtype=np.int32)), shape=(rows, items))


NOT_PD_LAYOUTS = [(20, 4), (9, 30)]  # (bad whole row, bad giant row): the lowest is found in the finish pass, then the main pass


@pytest.mark.gpu
@pytest.mark.parametrize("layout", NOT_PD_LAYOUTS, ids=["giant-lowest", "whole-lowest"])
@pytest.mark.parametrize("f", [80, 128], ids=["f80-wideT5", "f128-wideT8"])
def test_wide_cholesky_not_positive_definite_raises(lib, ctx, orc, f, layout):
    """_als.pyx:131-138 on the wide kernel: ValueError naming the lowest bad row, whether that row failed in the main
    pass or in the finish pass of a giant row; the next (good) half on the same context raises nothing."""
    items = 4000
    Y = factors(items, f, 3000 + f, 0.2)
    Cui = _indefinite_csr(items, *layout)
    lowest = min(layout)
    with pytest.raises(ValueError, match=rf"row {lowest}\b"):
        chol_truth(Cui, Y, 0.0)  # the fp64 truth agrees that the row is indefinite
    with pytest.raises(ValueError, match=rf"row {lowest}\b"):
        gpu_chol(lib, ctx, Cui, Y, 0.0)
    good = _indefinite_csr(items, -1, -1, seed=1)
    got = gpu_chol(lib, ctx, good, Y, 0.0)
    _check(*chol_bars(got, oracle_chol(orc, good, Y, 0.0), chol_truth(good, Y, 0.0), empty_rows(good)),
           f"good half after not-PD f={f}")


@pytest.mark.gpu
@pytest.mark.parametrize("f", [64, 80, 128], ids=["f64-NB4", "f80-wideT5", "f128-wideT8"])
def test_async_half_keeps_bad_row_until_status(lib, ctx, f):
    """The multi-GPU fit queues halves without reading bad_row back (als_least_squares_pregram_async) and collects
    failures with als_solver_status: a failed half followed by a good one must still be reported, with its row.

    Before this test the wide kernel (cholesky_wide.cu, T = 5..8) reset only bad_row[0] at the start of a half, so
    the good half erased the failure of the bad one and solver_status raised nothing at f = 80 and f = 128."""
    items = 4000
    Y = factors(items, f, 4000 + f, 0.2)
    bad, good = _indefinite_csr(items, 9, 30), _indefinite_csr(items, -1, -1, seed=1)
    dX = lib.DeviceFactors.from_host(ctx, np.zeros((48, f), np.float32))
    dY = lib.DeviceFactors.from_host(ctx, Y)
    Cb, Cg = lib.DeviceCSR.upload(ctx, bad), lib.DeviceCSR.upload(ctx, good)
    try:
        lib.gramian_shard(ctx, dY, 0, items)
        lib.half_pregram_async(ctx, Cb, dX, dY, 0.0, use_cg=False)
        lib.half_pregram_async(ctx, Cg, dX, dY, 0.0, use_cg=False)
        with pytest.raises(ValueError, match=r"row 9\b"):
            lib.solver_status(ctx)
        lib.half_pregram_async(ctx, Cg, dX, dY, 0.0, use_cg=False)
        lib.solver_status(ctx)  # a new collection period: nothing to report
    finally:
        for h in (Cb, Cg, dX, dY):
            h.close()


# ======================================================================================== c. CG half
CG_NARROW = [12, 20, 40, 64, 80, 96, 100, 127]  # ld 16, 32, ..., 128
CG_WIDE = [600, 700, 800, 1000, 1024]  # ld 640, 768, 896, 1024, 1024
CG_REG = 0.01


def _cg_case(small_matrix, f, orc):
    """A warm state: one oracle CG half from random factors, then the half under test starts from there."""
    Y = factors(small_matrix.shape[1], f, 5000 + f, 0.1)
    X = factors(small_matrix.shape[0], f, 6000 + f, 0.1)
    orc.least_squares_cg(small_matrix, X, Y, CG_REG, cg_steps=3)
    exp = X.copy()
    orc.least_squares_cg(small_matrix, exp, Y, CG_REG, cg_steps=3)
    return X, Y, exp, cg_truth(small_matrix, X, Y, CG_REG, 3)


_cg_cache = {}


def _cg_case_cached(small_matrix, f, orc):
    if f not in _cg_cache:
        _cg_cache.clear()
        _cg_cache[f] = _cg_case(small_matrix, f, orc)
    return _cg_cache[f]


@pytest.mark.gpu
@pytest.mark.parametrize("nv", [1, 2, 4], ids=["nv1", "nv2", "nv4"])
@pytest.mark.parametrize("f", CG_NARROW, ids=[f"f{f}-F{padded(f)}" for f in CG_NARROW])
def test_cg_half_narrow_width(lib, ctx, orc, small_matrix, f, nv):
    X, Y, exp, truth = _cg_case_cached(small_matrix, f, orc)
    with knob(ctx, "cg_nv", nv), Half(lib, ctx, small_matrix, X, Y) as h:
        got = h.cg(CG_REG)
    _check(*cg_bars(got, exp, truth, empty_rows(small_matrix)), f"cg f={f} (F={padded(f)}, NV={nv})")


@pytest.mark.gpu
@pytest.mark.parametrize("f", CG_WIDE, ids=[f"f{f}-F{padded(f)}" for f in CG_WIDE])
def test_cg_half_wide_width(lib, ctx, orc, small_matrix, f):
    X, Y, exp, truth = _cg_case_cached(small_matrix, f, orc)
    with Half(lib, ctx, small_matrix, X, Y) as h:
        got = h.cg(CG_REG)
    _check(*cg_bars(got, exp, truth, empty_rows(small_matrix)), f"cg f={f} (F={padded(f)})")


@pytest.mark.gpu
def test_cg_zero_steps_wide_leaves_factors(lib, ctx, small_matrix):
    """cg_steps = 0: the residual is formed and nothing moves (empty rows still become zero, _als.pyx:182-184)."""
    f = 700
    X, Y = factors(small_matrix.shape[0], f, 7, 0.1), factors(small_matrix.shape[1], f, 8, 0.1)
    with Half(lib, ctx, small_matrix, X, Y) as h:
        got = h.cg(CG_REG, steps=0)
    empty = empty_rows(small_matrix)
    assert np.all(got[empty] == 0)
    np.testing.assert_array_equal(got[~empty], X[~empty])


# ======================================================================================== d. loss
LOSS_WIDTHS = [8, 20, 40, 64, 72, 96, 100, 128, 250, 300, 500, 600, 700, 800, 1000]


@pytest.mark.gpu
@pytest.mark.parametrize("f", LOSS_WIDTHS, ids=[f"f{f}-ld{padded(f)}" for f in LOSS_WIDTHS])
def test_loss_width(lib, ctx, small_matrix, f):
    X, Y = factors(small_matrix.shape[0], f, 8000 + f, 0.1), factors(small_matrix.shape[1], f, 9000 + f, 0.1)
    with Half(lib, ctx, small_matrix, X, Y) as h:
        got = lib.calculate_loss(ctx, h.C, h.X, h.Y, 0.01)
    _check(*loss_bars(got, loss_truth(small_matrix, X, Y, 0.01)), f"loss f={f} (ld {padded(f)})")


# ======================================================================================== e. Gramian
GRAM_WIDTHS = [16, 24, 48, 57, 64, 72, 96, 100, 128, 640, 700, 896, 1000]
GRAM_ROWS = [1, 127, 128, 129, 5000]


def gram_input(rows, f, kind, seed):
    Y = factors(rows, f, seed, 0.3)
    if kind == "cancel":
        # odd columns are the even ones with the sign of the row alternating: their cross terms cancel pairwise
        s = np.where(np.arange(rows) % 2 == 0, 1.0, -1.0).astype(np.float32)[:, None]
        n = f // 2
        Y[:, 1:2 * n:2] = s * Y[:, 0:2 * n:2] * np.float32(1 + 1e-3)
        Y += np.float32(2.0)  # large common offset: sum of magnitudes >> the result
    return Y


def _gram_path(f, rows, knob_name):
    ld = padded(f)
    if knob_name:
        return knob_name
    if ld > 128:
        return f"wide{ld // 64}"
    return "tcgen05" if ld == 64 and rows >= 128 else f"fma{ld // 16}"


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mixed", "cancel"])
@pytest.mark.parametrize("rows", GRAM_ROWS, ids=[f"rows{r}" for r in GRAM_ROWS])
@pytest.mark.parametrize("f", GRAM_WIDTHS, ids=[f"f{f}-ld{padded(f)}" for f in GRAM_WIDTHS])
def test_gramian_width(lib, ctx, f, rows, kind):
    Y = gram_input(rows, f, kind, f * 7 + rows)
    d = lib.DeviceFactors.from_host(ctx, Y)
    G = lib.gramian(ctx, d)
    d.close()
    _check(*gram_bars(G, Y), f"gramian f={f} rows={rows} {kind} ({_gram_path(f, rows, None)})")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mixed", "cancel"])
@pytest.mark.parametrize("rows", GRAM_ROWS, ids=[f"rows{r}" for r in GRAM_ROWS])
@pytest.mark.parametrize("name", ["gramian_mma", "gramian_fma"])
@pytest.mark.parametrize("f", [16, 48, 64])
def test_gramian_knobs(lib, ctx, f, name, rows, kind):
    Y = gram_input(rows, f, kind, f * 11 + rows)
    d = lib.DeviceFactors.from_host(ctx, Y)
    with knob(ctx, name, 1):
        G = lib.gramian(ctx, d)
    d.close()
    _check(*gram_bars(G, Y), f"gramian f={f} rows={rows} {kind} ({name})")


# ======================================================================================== f. knob equivalence
KNOB_SETTINGS = [("short_max", 0), ("short_max", 16), ("short_max", 32), ("short_max", 48), ("short_serial", 1),
                 ("whiten_fma", 1)]


@pytest.mark.gpu
@pytest.mark.parametrize("setting", KNOB_SETTINGS, ids=[f"{n}={v}" for n, v in KNOB_SETTINGS])
@pytest.mark.parametrize("f", [32, 40, 64])
def test_cholesky_knobs_change_nothing(lib, ctx, orc, chol_matrix, f, setting):
    """The short-row knobs move rows between the n x n push-through kernels and the full-size kernel; every setting
    must meet the fp64 bars.  (4000 items: the short rows are numerous enough for the push-through path to run at
    every short_max > 0.)"""
    Y, exp, truth = _chol_case(chol_matrix, f, 0.01, orc)
    lens = np.diff(chol_matrix.indptr)
    if setting[0] == "short_max" and setting[1]:
        assert (lens <= setting[1]).sum() * 16 >= chol_matrix.shape[1]  # cholesky.cu: the path pays off, so it runs
    with knob(ctx, *setting):
        got = gpu_chol(lib, ctx, chol_matrix, Y, 0.01)
    _check(*chol_bars(got, exp, truth, empty_rows(chol_matrix)), f"cholesky f={f} {setting[0]}={setting[1]}")


@pytest.mark.gpu
@pytest.mark.parametrize("f", [32, 40, 64, 100])
def test_cholesky_half_is_deterministic(lib, ctx, chol_matrix, f):
    """Two runs on the same handles give the same bits: the aux-stream overlap of the short-row kernels, the deferred
    list and the order in which the chunk partials of giant rows are summed do not depend on scheduling."""
    Y = factors(chol_matrix.shape[1], f, 1000 + f, 0.2)
    with Half(lib, ctx, chol_matrix, np.zeros((chol_matrix.shape[0], f), np.float32), Y) as h:
        a = h.chol(0.01)
        b = h.chol(0.01)
    print(f"cholesky f={f} twice: {int((a != b).sum())} differing values")
    np.testing.assert_array_equal(a, b)


# ======================================================================================== g. top-k
TOPK_WIDTHS = [1, 17, 80, 700, 1024]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 10])
@pytest.mark.parametrize("f", TOPK_WIDTHS, ids=[f"f{f}-{'sort' if f > 128 else 'F' + str(padded(f))}" for f in TOPK_WIDTHS])
def test_topk_width(lib, ctx, orc, f, k):
    from implicit_b200 import synthetic

    items, q = factors(3000, f, 10 * f + k, 0.3), factors(150, f, 10 * f + k + 1, 0.3)
    liked = synthetic.power_law_csr(150, 3000, 2500, 8)
    filt = np.array([0, 5, 17, 2999])
    di, dq, dl = lib.DeviceFactors.from_host(ctx, items), lib.DeviceFactors.from_host(ctx, q), lib.DeviceCSR.upload(ctx, liked)
    ids, sc = lib.topk(ctx, di, dq, k, liked=dl, filter_items=filt)
    for h in (di, dq, dl):
        h.close()
    eids, esc = orc.topk(items, q, k, filter_query_items=liked, filter_items=filt)
    _check(*topk_bars(ids, sc, eids, esc, q, items, filt), f"topk f={f} k={k}")
    liked_hit = [np.isin(ids[r], liked.indices[liked.indptr[r]:liked.indptr[r + 1]]).any() for r in range(150)]
    assert not any(liked_hit)
