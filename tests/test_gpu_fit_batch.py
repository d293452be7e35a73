"""GPU suite (-m gpu): the final models of many fits in one launch (pareben_fit_batch, Problem.fit_batch, EBelasticNetMulti).

Each record of a batch must be bitwise the model pareben_fit returns for that fit alone: support, candidate ids, beta,
variance, Wald score, intercepts, residual variance / log-likelihood and status, for every kernel variant (Gaussian main
effects with the Gram organisation on and off, Gaussian Epis, both binomial contractions, binomial Epis, streaming
mode).  Fold models must agree with pareben_run_fits and with the reference C.  The Gram work test counts the fits of
a call, so every comparison with a single-fit call pins PAREBEN_GRAM.
"""
import ctypes

import numpy as np
import pytest

from oracle import rlayer as R
from record_layout import expand

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pb(built):
    import pareben_b200 as pb
    if pb.device_count() < 1:
        pytest.fail("no CUDA device: the -m gpu suite must run on the B200 box")
    return pb


def _responses(y, n_extra, seed):
    rng = np.random.default_rng(seed)
    return np.column_stack([y] + [rng.permutation(y) for _ in range(n_extra)])


def _points(pb, X, Y, epis, a_idx, l_idx):
    """One (alpha, lambda) per response: response t at row l_idx[t] * 20 + a_idx[t] of its own BuildGrid grid."""
    A, L = [], []
    for t in range(Y.shape[1]):
        g = pb.BuildGrid(X, Y[:, t], 0, "yes" if epis else "no")
        r = l_idx[t] * 20 + a_idx[t]
        A.append(g["alpha"][r]); L.append(g["lambda"][r])
    return np.array(A), np.array(L)


def _same_record(r, i, q, j):
    for key in ("n_effects", "cand", "beta", "var", "scalars", "status", "fold_err"):
        assert np.array_equal(r[key][i], q[key][j]), f"record {i}: {key} differs"


def _check_against_fit(pb, X, Y, A, L, epis, prior):
    """One fit per response in one batch, each record against pareben_fit on a problem holding that response alone."""
    gaussian = prior == "gaussian"
    T, k = Y.shape[1], X.shape[1]
    with pb.Problem(X, Y, None, 0, epis, prior) as p:
        r = p.fit_batch(np.arange(T), np.zeros(T), A, L)
        info = p.contraction_info()
    assert r["cand"].shape[1] >= r["n_effects"].max()
    for t in range(T):
        with pb.Problem(X, Y[:, t], None, 0, epis, prior) as q:
            table, wald, icpt, extra, st = q.fit(A[t], L[t])
        got = expand(r["n_effects"][t], r["cand"][t], r["beta"][t], r["var"][t], k, epis, gaussian)
        assert np.array_equal(got, table), f"response {t}: table differs"
        assert np.array_equal(r["scalars"][t], [wald, icpt[0], icpt[1], extra]), f"response {t}: scalars differ"
        assert r["status"][t] == st and r["fold_err"][t] == 0
        if gaussian and epis:
            assert r["n_effects"][t] == np.count_nonzero(table[:, 4])
        assert not r["beta"][t, r["n_effects"][t]:].any() and not r["cand"][t, r["n_effects"][t]:].any()
    return r, info


@pytest.mark.parametrize("gram", ["0", "1"])
def test_gaussian_main_effects_bundled(pb, bundled, monkeypatch, gram):
    monkeypatch.setenv("PAREBEN_GRAM", gram)
    X, Y = bundled["BASIS"], _responses(bundled["y"], 5, 101)
    A, L = _points(pb, X, Y, False, [0, 19, 0, 10, 5, 0], [19, 0, 18, 2, 15, 8])
    r, _ = _check_against_fit(pb, X, Y, A, L, False, "gaussian")
    assert r["n_effects"].max() >= 8 * max(1, r["n_effects"].min()), r["n_effects"]      # strides of very different fill


def test_gaussian_epis_cached(pb, bundled, monkeypatch):
    monkeypatch.setenv("PAREBEN_GRAM", "1")
    X, Y = bundled["BASIS"][:300, :40], _responses(bundled["y"][:300], 3, 103)
    A, L = _points(pb, X, Y, True, [0, 10, 19, 0], [19, 0, 12, 6])
    _check_against_fit(pb, X, Y, A, L, True, "gaussian")


def test_binomial_main_effects_tensor_core(pb, bundled):
    X, Y = bundled["BASISbinomial"], _responses(bundled["yBinomial"], 4, 107)
    A, L = _points(pb, X, Y, False, [0, 19, 0, 10, 5], [19, 0, 17, 4, 12])
    r, (tc, n_tc) = _check_against_fit(pb, X, Y, A, L, False, "binomial")
    assert tc and n_tc > 0, "genotype codes must take the int8 tensor-core contraction"
    assert r["n_effects"].max() > r["n_effects"].min()


def test_binomial_main_effects_real_valued(pb, bundled):
    rng = np.random.default_rng(109)
    X = bundled["BASISbinomial"][:, :150] + rng.normal(0, 0.25, (500, 150))
    Y = _responses(bundled["yBinomial"], 3, 113)
    A, L = _points(pb, X, Y, False, [0, 19, 6, 0], [19, 0, 10, 15])
    _, (tc, _n) = _check_against_fit(pb, X, Y, A, L, False, "binomial")
    assert not tc


def test_binomial_epis(pb, bundled):
    X, Y = bundled["BASISbinomial"][:200, :30], _responses(bundled["yBinomial"][:200], 3, 127)
    A, L = _points(pb, X, Y, True, [0, 19, 10, 0], [19, 0, 12, 6])
    _check_against_fit(pb, X, Y, A, L, True, "binomial")


def test_gaussian_streaming_config5_slice(pb):
    from pareben_b200.synth import config5
    d = config5(1000, 2000)
    X, Y = d["X"].astype(np.float64), _responses(d["y"], 2, 131)
    A, L = _points(pb, X, Y, True, [0, 19, 10], [8, 0, 4])
    pb.set_mode(pb.MODE_STREAMING)
    try:
        with pb.Problem(X[:50], Y[:50], None, 0, True, "gaussian") as p:
            assert p.streaming
        _check_against_fit(pb, X, Y, A, L, True, "gaussian")
    finally:
        pb.set_mode(pb.MODE_AUTO)


def test_basis_cap_fit(pb, bundled, monkeypatch):
    """A fit that ends at the basis cap next to one that does not; the record stride is the (low) cap."""
    monkeypatch.setenv("PAREBEN_GRAM", "0")
    monkeypatch.setenv("PAREBEN_BASIS_CAP", "6")
    X, Y = bundled["BASIS"], _responses(bundled["y"], 1, 137)
    A, L = _points(pb, X, Y, False, [0, 0], [19, 0])
    with pb.Problem(X, Y, None, 0) as p:
        assert p.max_effects() == 6
    r, _ = _check_against_fit(pb, X, Y, A, L, False, "gaussian")
    assert r["status"][0] & pb.FIT_BASIS_CAP and r["n_effects"][0] == 6
    assert not r["status"][1] & pb.FIT_BASIS_CAP


@pytest.mark.parametrize("prior", ["gaussian", "binomial"])
def test_batch_composition_does_not_matter(pb, bundled, monkeypatch, prior):
    """The same fit alone and inside a shuffled batch of 300 (a regularisation path of one response, plus two other
    responses) gives bitwise the same record (cached kernels)."""
    monkeypatch.setenv("PAREBEN_GRAM", "0")
    if prior == "gaussian":
        X, Y = bundled["BASIS"], _responses(bundled["y"], 2, 139)
    else:
        X, Y = bundled["BASISbinomial"], _responses(bundled["yBinomial"], 2, 149)
    grids = [pb.BuildGrid(X, Y[:, t]) for t in range(3)]
    rows = np.arange(0, 400, 4)                                          # 100 grid points per response
    target = np.repeat(np.arange(3), rows.size)
    alpha = np.concatenate([g["alpha"][rows] for g in grids])
    lam = np.concatenate([g["lambda"][rows] for g in grids])
    rng = np.random.default_rng(151)
    order = rng.permutation(target.size)
    with pb.Problem(X, Y, None, 0, False, prior) as p:
        r = p.fit_batch(target[order], np.zeros(order.size), alpha[order], lam[order])
        order2 = rng.permutation(target.size)
        r2 = p.fit_batch(target[order2], np.zeros(order2.size), alpha[order2], lam[order2])
        pos = np.empty_like(order2); pos[order2] = np.arange(order2.size)
        for i in range(order.size):
            _same_record(r, i, r2, pos[order[i]])
        for i in rng.choice(order.size, 12, replace=False):
            alone = p.fit_batch(target[order[i]:order[i] + 1], np.zeros(1), alpha[order[i]:order[i] + 1], lam[order[i]:order[i] + 1])
            _same_record(r, i, alone, 0)
    assert r["n_effects"].max() > 4 * max(1, r["n_effects"].min())


@pytest.mark.parametrize("prior", ["gaussian", "binomial"])
def test_fold_models(pb, bundled, monkeypatch, prior):
    """Fold fits: fold error, status and support size equal pareben_run_fits bitwise; the models equal the reference C
    run on the fold's training rows at the boundary tests' tolerances."""
    monkeypatch.setenv("PAREBEN_GRAM", "0")
    from pareben_b200.cross_validate import _record_weight
    if prior == "gaussian":
        X, Y, rtol = bundled["BASIS"][:300, :80], _responses(bundled["y"][:300], 1, 157), 1e-8
    else:
        X, Y, rtol = bundled["BASISbinomial"][:, :80], _responses(bundled["yBinomial"], 1, 163), 5e-8
    folds = pb.AssignToFolds(X, 3)
    grids = [pb.BuildGrid(X, Y[:, t]) for t in range(2)]
    rows = [45, 250, 390]
    target = np.repeat(np.arange(2), 3 * len(rows))
    fold = np.tile(np.repeat(np.arange(1, 4), len(rows)), 2)
    alpha = np.concatenate([np.tile(g["alpha"][rows], 3) for g in grids])
    lam = np.concatenate([np.tile(g["lambda"][rows], 3) for g in grids])
    with pb.Problem(X, Y, folds, 3, False, prior) as p:
        r = p.fit_batch(target, fold, alpha, lam)
        err, st, ns, _it = p.run_fits(fold, alpha, lam, target)
    assert np.array_equal(r["fold_err"], err) and np.array_equal(r["status"], st)
    assert np.array_equal((r["beta"] != 0).sum(axis=1), ns)
    lib = R.fit_lib(R.available_kind())
    n_tr = X.shape[0] - np.bincount(folds)[1:]
    for i in range(target.size):
        e, fit = R.fit_one(X, Y[:, target[i]], folds, fold[i], lam[i], alpha[i], prior=prior, lib=lib)
        got = _record_weight(r["n_effects"][i], r["cand"][i], r["beta"][i], r["var"][i], False, prior == "gaussian", X.shape[1],
                             n_tr[fold[i] - 1])
        want = fit.weight
        assert got.shape == want.shape and np.array_equal(got[:, :2], want[:, :2]), f"fit {i}: support differs"
        for c in (2, 3):
            assert np.allclose(got[:, c], want[:, c], rtol=rtol, atol=1e-14), f"fit {i}: column {c}"
        assert abs(r["fold_err"][i] - e) <= rtol * abs(e)


def _same_result(a, b):
    assert set(a) == set(b)
    for key in a:
        if isinstance(a[key], np.ndarray):
            assert np.array_equal(a[key], b[key]), key
        else:
            assert a[key] == b[key], key


@pytest.mark.parametrize("prior", ["gaussian", "binomial"])
@pytest.mark.parametrize("epis", ["no", "yes"])
def test_ebelasticnet_multi_equals_per_column(pb, bundled, monkeypatch, prior, epis):
    monkeypatch.setenv("PAREBEN_GRAM", "1")
    if prior == "gaussian":
        X, Y = (bundled["BASIS"][:300, :40], _responses(bundled["y"][:300], 2, 167)) if epis == "yes" else \
               (bundled["BASIS"], _responses(bundled["y"], 2, 167))
    else:
        X, Y = (bundled["BASISbinomial"][:200, :30], _responses(bundled["yBinomial"][:200], 2, 173)) if epis == "yes" else \
               (bundled["BASISbinomial"], _responses(bundled["yBinomial"], 2, 173))
    A, L = _points(pb, X, Y, epis == "yes", [0, 10, 19], [19, 5, 10])
    multi = pb.EBelasticNetMulti(X, Y, L, A, Epis=epis, prior=prior)
    single = pb.EBelasticNet_Gaussian if prior == "gaussian" else pb.EBelasticNet_Binomial
    assert len(multi) == 3
    for t in range(3):
        _same_result(multi[t], single(X, Y[:, t], L[t], A[t], epis))
    broadcast = pb.EBelasticNetMulti(X, Y, L[0], A[0], Epis=epis, prior=prior)         # scalars apply to every response
    _same_result(broadcast[0], multi[0])


def test_errors(pb, bundled):
    X, Y = bundled["BASIS"][:100, :20], _responses(bundled["y"][:100], 2, 179)
    folds = pb.AssignToFolds(X, 3)
    lib = pb.load()
    ip, dp = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_double)
    with pb.Problem(X, Y, None, 0) as p:
        me = p.max_effects()
        assert me >= 1
        t, f, a, lam = np.arange(3, dtype=np.int32), np.zeros(3, np.int32), np.ones(3), np.full(3, 0.5)
        ne, cand = np.full(3, -7, np.int32), np.full(3 * me, -7, np.int32)
        beta, var, sc, st, fe = np.full(3 * me, -7.0), np.full(3 * me, -7.0), np.full(12, -7.0), np.full(3, -7, np.int32), np.full(3, -7.0)

        def call(m, tt, ff, width):
            return lib.pareben_fit_batch(p._h, m, tt.ctypes.data_as(ip), ff.ctypes.data_as(ip), a.ctypes.data_as(dp),
                                         lam.ctypes.data_as(dp), width, ne.ctypes.data_as(ip), cand.ctypes.data_as(ip),
                                         beta.ctypes.data_as(dp), var.ctypes.data_as(dp), sc.ctypes.data_as(dp),
                                         st.ctypes.data_as(ip), fe.ctypes.data_as(dp))
        assert call(3, t, f, me - 1) == -1                                      # max_effects below pareben_max_effects
        assert call(3, np.array([0, 1, 3], np.int32), f, me) == -1              # target out of range
        assert call(3, t, np.array([0, 0, 1], np.int32), me) == -1              # fold 1 on a problem without folds
        assert call(0, t, f, me) == 0                                           # n_fits = 0: a no-op
        assert (ne == -7).all() and (cand == -7).all() and (beta == -7).all() and (sc == -7).all() and (fe == -7).all()
        assert lib.pareben_fit_batch(p._h, 0, None, None, None, None, 0, None, None, None, None, None, None, None) == 0
        empty = p.fit_batch([], [], [], [])
        assert empty["n_effects"].size == 0 and empty["cand"].shape == (0, me)
        with pytest.raises(pb.ParebenError):
            p.fit(1.0, 1.0)                                                     # pareben_fit: one response only
    with pb.Problem(X, Y, folds, 3) as p:
        with pytest.raises(pb.ParebenError):
            p.fit_batch([0], [0], [1.0], [0.5])                                 # fold 0 on a problem with folds
        with pytest.raises(pb.ParebenError):
            p.fit_batch([0], [4], [1.0], [0.5])                                 # fold label out of range
        with pytest.raises(pb.ParebenError):
            p.fit_batch([0, 3], [1, 1], [1.0, 1.0], [0.5, 0.5])                 # target out of range
