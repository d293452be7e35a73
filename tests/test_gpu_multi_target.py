"""GPU suite (-m gpu): several responses against one design in one call (pareben_*_multi, CrossValidateMulti).

Every fit of a multi-response call must be bitwise the same fit of a single-response call: fold error, status, support
size and outer iterations, for every kernel variant (Gaussian / binomial, main effects / Epis, the int8 tensor-core and
FP64 binomial contractions, the Gram organisation on and off, streaming mode).  The Gram work test counts the fits of
the whole call, so the comparisons pin PAREBEN_GRAM: with it pinned, both calls take the same organisation.
"""
import ctypes

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pb(built):
    import pareben_b200 as pb
    if pb.device_count() < 1:
        pytest.fail("no CUDA device: the -m gpu suite must run on the B200 box")
    return pb


def _responses(y, n_extra, seed):
    """y and n_extra seeded permutations of it, as columns."""
    rng = np.random.default_rng(seed)
    return np.column_stack([y] + [rng.permutation(y) for _ in range(n_extra)])


def _sub_grids(pb, X, Y, epis, a_idx, l_idx):
    """(T, n_grid) alpha and lambda: each response's BuildGrid grid (from its own lambda_max), rows a_idx x l_idx."""
    rows = (np.asarray(l_idx)[:, None] * 20 + np.asarray(a_idx)[None, :]).ravel()
    grids = [pb.BuildGrid(X, Y[:, t], 0, "yes" if epis else "no") for t in range(Y.shape[1])]
    return np.stack([g["alpha"][rows] for g in grids]), np.stack([g["lambda"][rows] for g in grids])


def _compare(pb, X, Y, n_folds, A, L, epis, prior):
    """Multi-response tables (run_fits with targets, and cv_grid_multi) against one single-response problem per column."""
    folds = pb.AssignToFolds(X, n_folds)
    T, n_grid = A.shape
    fold = np.tile(np.arange(1, n_folds + 1), n_grid).astype(np.int32)
    with pb.Problem(X, Y, folds, n_folds, epis, prior) as p:
        assert p.n_targets == T
        target = np.repeat(np.arange(T), n_grid * n_folds).astype(np.int32)
        multi = p.run_fits(np.tile(fold, T), np.repeat(A, n_folds, axis=1).ravel(), np.repeat(L, n_folds, axis=1).ravel(), target)
        grid_multi = p.cv_grid_multi(A, L)
        info = p.contraction_info()
    for t in range(T):
        with pb.Problem(X, Y[:, t], folds, n_folds, epis, prior) as q:
            single = q.run_fits(fold, np.repeat(A[t], n_folds), np.repeat(L[t], n_folds))
            grid_single = q.cv_grid(A[t], L[t])
        sl = slice(t * n_grid * n_folds, (t + 1) * n_grid * n_folds)
        for name, m, s in zip(("fold error", "status", "support size", "iterations"), multi, single):
            assert np.array_equal(m[sl], s), f"response {t}: {name} differs"
        for m, s in zip(grid_multi, grid_single):
            assert np.array_equal(m[t], s)
        assert np.array_equal(grid_multi[0][t].ravel(), single[0])
    return multi, info


@pytest.mark.parametrize("gram", ["1", "0"])
def test_gaussian_main_effects_bundled(pb, bundled, monkeypatch, gram):
    monkeypatch.setenv("PAREBEN_GRAM", gram)
    X, Y = bundled["BASIS"], _responses(bundled["y"], 2, 7)
    A, L = _sub_grids(pb, X, Y, False, np.arange(0, 20, 2), np.arange(0, 20, 2))
    multi, _ = _compare(pb, X, Y, 5, A, L, False, "gaussian")
    assert (multi[2] > 0).any()
    with pb.Problem(X, Y, pb.AssignToFolds(X, 5), 5, False, "gaussian") as p:
        p.run_fits(np.array([1, 2], np.int32), A[0, :2], L[0, :2], np.array([0, 2], np.int32))
        assert p.gram_info()[0] == (gram == "1")


def test_gaussian_epis_cached(pb, bundled, monkeypatch):
    monkeypatch.setenv("PAREBEN_GRAM", "1")
    X, Y = bundled["BASIS"][:300, :40], _responses(bundled["y"][:300], 2, 11)
    A, L = _sub_grids(pb, X, Y, True, [0, 5, 10, 19], [0, 4, 8, 12, 16])
    _compare(pb, X, Y, 3, A, L, True, "gaussian")


def test_binomial_main_effects_tensor_core(pb, bundled):
    X, Y = bundled["BASISbinomial"], _responses(bundled["yBinomial"], 2, 13)
    A, L = _sub_grids(pb, X, Y, False, np.arange(0, 20, 2), np.arange(0, 20, 2))
    _, (tc, n_tc) = _compare(pb, X, Y, 5, A, L, False, "binomial")
    assert tc and n_tc > 0, "genotype codes must take the int8 tensor-core contraction"


def test_binomial_main_effects_real_valued(pb, bundled):
    rng = np.random.default_rng(17)
    X = bundled["BASISbinomial"][:, :150] + rng.normal(0, 0.25, (500, 150))
    Y = _responses(bundled["yBinomial"], 2, 19)
    A, L = _sub_grids(pb, X, Y, False, [0, 6, 12, 19], [0, 5, 10, 15, 19])
    _, (tc, _n) = _compare(pb, X, Y, 5, A, L, False, "binomial")
    assert not tc


def test_binomial_epis(pb, bundled):
    X, Y = bundled["BASISbinomial"][:200, :30], _responses(bundled["yBinomial"][:200], 2, 23)
    A, L = _sub_grids(pb, X, Y, True, [0, 10, 19], [0, 6, 12, 18])
    _compare(pb, X, Y, 3, A, L, True, "binomial")


def test_gaussian_streaming_config5_slice(pb):
    from pareben_b200.synth import config5
    d = config5(1000, 2000)
    X, Y = d["X"].astype(np.float64), _responses(d["y"], 2, 29)
    A, L = _sub_grids(pb, X, Y, True, [0, 10, 19], [0, 4, 8])
    pb.set_mode(pb.MODE_STREAMING)
    try:
        with pb.Problem(X[:50], Y[:50], pb.AssignToFolds(X[:50], 2), 2, True, "gaussian") as p:
            assert p.streaming
        _compare(pb, X, Y, 3, A, L, True, "gaussian")
    finally:
        pb.set_mode(pb.MODE_AUTO)


@pytest.mark.parametrize("epis", [False, True])
@pytest.mark.parametrize("T", [1, 5, 17])
def test_lambda_max_multi_bitwise(pb, bundled, epis, T):
    """17 responses cross a 16-response tile of the kernel."""
    X = bundled["BASIS"][:, :60] if epis else bundled["BASIS"]
    Y = _responses(bundled["y"], T - 1, 31)
    with pb.Problem(X, Y, None, 0, epis) as p:
        lm = p.lambda_max_multi()
    assert lm.shape == (T,)
    for t in range(T):
        with pb.Problem(X, Y[:, t], None, 0, epis) as q:
            assert lm[t] == q.lambda_max(), f"response {t}"


def _same_result(a, b):
    assert set(a) == set(b)
    for key in a:
        if isinstance(a[key], dict):
            _same_result(a[key], b[key])
        elif isinstance(a[key], np.ndarray):
            assert np.array_equal(a[key], b[key]), key
        else:
            assert a[key] == b[key], key


@pytest.mark.filterwarnings("ignore::RuntimeWarning")       # status reports of _which_min: not what this checks
@pytest.mark.parametrize("prior", ["gaussian", "binomial"])
@pytest.mark.parametrize("search", ["global", "local"])
def test_cross_validate_multi_equals_per_column(pb, bundled, monkeypatch, prior, search):
    monkeypatch.setenv("PAREBEN_GRAM", "1")
    if prior == "gaussian":
        X, Y = bundled["BASIS"][:400, :120], _responses(bundled["y"][:400], 1, 37)
    else:
        X, Y = bundled["BASISbinomial"][:, :120], _responses(bundled["yBinomial"], 1, 41)
    multi = pb.CrossValidateMulti(X, Y, 3, Epis="no", prior=prior, search=search)
    assert len(multi) == 2
    for t in range(2):
        _same_result(multi[t], pb.CrossValidate(X, Y[:, t], 3, Epis="no", prior=prior, search=search))


def test_shards_sum_to_the_whole_table(pb, bundled):
    X, Y = bundled["BASISbinomial"][:, :200], _responses(bundled["yBinomial"], 2, 43)
    folds = pb.AssignToFolds(X, 5)
    A, L = _sub_grids(pb, X, Y, False, [0, 7, 14, 19], [0, 5, 10, 15])
    whole = pb.cv_grid_multi(X, Y, folds, 5, A, L, prior="binomial")
    parts = [pb.cv_grid_multi(X, Y, folds, 5, A, L, prior="binomial", shard=s, n_shards=3) for s in range(3)]
    for i in range(3):
        assert np.array_equal(sum(p[i] for p in parts), whole[i])
    # the shard rule is pareben_shard_plan on the flattened (response, grid point) rows: other entries stay 0
    for s in range(3):
        others = np.ones(whole[0].size, bool)
        others[pb.shard_plan(L.ravel(), 5, s, 3)] = False
        assert not parts[s][0].ravel()[others].any()
    if pb.device_count() >= 2:
        two = pb.cv_grid_multi(X, Y, folds, 5, A, L, prior="binomial", n_devices=2)
        for i in range(3):
            assert np.array_equal(two[i], whole[i])


def test_errors(pb, bundled):
    X, y = bundled["BASIS"][:100, :20], bundled["y"][:100]
    Y = _responses(y, 2, 47)
    folds = pb.AssignToFolds(X, 3)
    with pytest.raises(ValueError):
        pb.Problem(X, Y[:99], folds, 3)
    with pytest.raises(ValueError):
        pb.Problem(X, Y[:, :0], folds, 3)
    with pytest.raises(ValueError):
        pb.cv_grid_multi(X, Y, folds, 3, np.ones((2, 4)), np.ones((2, 4)))          # 3 responses, grids for 2
    lib = pb.load()
    h = ctypes.c_void_p()
    Xf, Yf = np.asfortranarray(X), np.asfortranarray(Y)
    dp = ctypes.POINTER(ctypes.c_double)
    rc = lib.pareben_problem_create_multi(ctypes.byref(h), 0, Xf.ctypes.data_as(dp), 100, 20, Yf.ctypes.data_as(dp), 0,
                                          folds.ctypes.data_as(ctypes.POINTER(ctypes.c_int)), 3, 0, 0)
    assert rc == -1                                                                   # PAREBEN_EINVAL: n_targets < 1
    with pb.Problem(X, Y, folds, 3) as p:
        with pytest.raises(pb.ParebenError):
            p.lambda_max()
        with pytest.raises(pb.ParebenError):
            p.sl_filter(0.02, 0.05)
        with pytest.raises(pb.ParebenError):
            p.cv_grid(np.ones(2), np.ones(2))
        with pytest.raises(pb.ParebenError):
            p.run_fits(np.array([1], np.int32), np.ones(1), np.ones(1), np.array([3], np.int32))
    with pb.Problem(X, Y, None, 0) as p:
        with pytest.raises(pb.ParebenError):
            p.fit(1.0, 1.0)
