"""GPU suite (-m gpu), part 4: the Gram organisation of the Gaussian cached kernels.

The candidate-cache row of a basis depends on the fold alone, so the library builds the rows of every candidate once per
fold (fold_gram_kernel) and all fits of the fold share them; PAREBEN_GRAM=0 keeps the reference's organisation (one cache
per fit, recomputed by every add and at the top of every outer iteration).  Both must give the same tables -- the same
sums in a different summation order -- and both are checked against the oracle by the other GPU tests (which run with
whichever organisation the work test picks).  The main-effect test reaches active sets of about 230, so its fits run
the register and 8-wide panel paths of the SPD inverse and both forms of the quadratic forms; those kernels are tested
on their own, at every path boundary, in test_gpu_linalg_kernels.py.
"""
import os

import numpy as np
import pytest

from oracle import rlayer as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pb(built):
    import pareben_b200 as pb
    if pb.device_count() < 1:
        pytest.fail("no CUDA device: the -m gpu suite must run on the B200 box")
    return pb


def _both(pb, X, y, folds, n_folds, epis, fold, a, l):
    out = {}
    old = os.environ.get("PAREBEN_GRAM")
    try:
        for mode in ("0", "1"):
            os.environ["PAREBEN_GRAM"] = mode
            with pb.Problem(X, y, folds, n_folds, epis, "gaussian") as p:
                err, st, ns, it = p.run_fits(fold, a, l)
                in_use, avoided, build_ms = p.gram_info()
                assert in_use == (mode == "1")
                assert (avoided > 0) == (mode == "1")
                err2, st2, ns2, it2 = p.run_fits(fold, a, l)          # second call: the matrices exist, nothing is rebuilt
                assert p.gram_info()[2] == 0.0
                assert np.array_equal(err, err2) and np.array_equal(ns, ns2)
                out[mode] = (err, st, ns, it)
    finally:
        if old is None:
            os.environ.pop("PAREBEN_GRAM", None)
        else:
            os.environ["PAREBEN_GRAM"] = old
    return out


def test_gram_matches_per_fit_cache_main_effects(pb, bundled):
    """Bundled 1000 x 481 Gaussian design, 10 folds, every 9th fit of the 4,000 (active sets up to ~230: the register
    and 8-wide panel paths of the SPD inverse, SIMT and tensor-core quadratic forms)."""
    X, y, nf = bundled["BASIS"].astype(np.float64), bundled["y"], 10
    folds = pb.AssignToFolds(X, nf)
    grid = pb.BuildGrid(X, y, nf)
    fold = np.tile(np.arange(1, nf + 1), 400); a = np.repeat(grid["alpha"], nf); l = np.repeat(grid["lambda"], nf)
    sel = np.arange(0, fold.size, 9)
    out = _both(pb, X, y, folds, nf, False, fold[sel].astype(np.int32), a[sel], l[sel])
    (e0, s0, n0, i0), (e1, s1, n1, i1) = out["0"], out["1"]
    assert np.all(s0 == 0) and np.all(s1 == 0)
    assert np.array_equal(n0, n1) and np.array_equal(i0, i1)
    assert n0.max() > 150
    assert np.max(np.abs(e1 - e0) / np.abs(e0)) < 1e-10
    # and against the oracle on the cheapest and the most expensive of them
    lib = R.fit_lib(R.available_kind())
    for i in (int(np.argmax(n1)), int(np.argmin(n1))):
        e, fit = R.fit_one(X, y, folds, int(fold[sel][i]), l[sel][i], a[sel][i], False, "gaussian", lib)
        assert abs(e1[i] - e) / abs(e) < 1e-8


def test_gram_matches_per_fit_cache_epis(pb):
    """Pair candidates generated on the fly: K = 40 loci -> 820 candidates, 3 folds."""
    rng = np.random.default_rng(20261019)
    n, k, nf = 240, 40, 3
    X = rng.choice([-1.0, 0.0, 1.0], size=(n, k), p=[0.25, 0.5, 0.25])
    y = 1.5 * X[:, 3] - 1.0 * X[:, 7] * X[:, 21] + 0.8 * X[:, 30] + rng.normal(0, 1.0, n)
    folds = pb.AssignToFolds(X, nf)
    grid = pb.BuildGrid(X, y, nf, "yes")
    rows = np.arange(0, 400, 7)
    fold = np.tile(np.arange(1, nf + 1), rows.size).astype(np.int32); a = np.repeat(grid["alpha"][rows], nf); l = np.repeat(grid["lambda"][rows], nf)
    out = _both(pb, X, y, folds, nf, True, fold, a, l)
    (e0, s0, n0, i0), (e1, s1, n1, i1) = out["0"], out["1"]
    assert np.array_equal(s0, s1) and np.array_equal(n0, n1) and np.array_equal(i0, i1)
    assert np.max(np.abs(e1 - e0) / np.abs(e0)) < 1e-10
    assert n1.max() >= 3
    # (parity of Epis fits with the oracle: tests/test_gpu_shapes.py, which runs with the Gram organisation)


def test_gram_is_skipped_when_the_call_is_too_small(pb):
    """One fit of a 1,500-candidate problem does not pay for 1,500 cache rows: the work test leaves the per-fit cache on,
    and a later big call on the same handle switches over -- with the same result for the fit both calls share."""
    rng = np.random.default_rng(7)
    n, k, nf = 150, 1500, 2
    X = rng.choice([-1.0, 0.0, 1.0], size=(n, k), p=[0.25, 0.5, 0.25])
    y = X[:, 5] - 0.7 * X[:, 900] + rng.normal(0, 1.0, n)
    folds = pb.AssignToFolds(X, nf)
    grid = pb.BuildGrid(X, y, nf)
    rows = np.arange(100, 400, 15)
    old = os.environ.pop("PAREBEN_GRAM", None)
    try:
        with pb.Problem(X, y, folds, nf, False, "gaussian") as p:
            e_one, st, ns_one, _ = p.run_fits(np.array([1], np.int32), grid["alpha"][rows[:1]], grid["lambda"][rows[:1]])
            assert p.gram_info()[0] is False
            fold = np.tile(np.arange(1, nf + 1), rows.size).astype(np.int32)
            e_all, st, ns_all, _ = p.run_fits(fold, np.repeat(grid["alpha"][rows], nf), np.repeat(grid["lambda"][rows], nf))
            assert p.gram_info()[0] is True and p.gram_info()[2] > 0
            assert ns_all[0] == ns_one[0] and abs(e_all[0] - e_one[0]) <= 1e-10 * abs(e_one[0])
    finally:
        if old is not None:
            os.environ["PAREBEN_GRAM"] = old
