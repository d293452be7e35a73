"""CPU suite, part 1: the oracle itself is pinned before anything trusts it.
 * R RNG emulator against R's documented known answers.
 * R-layer restatement against the CrossValidate output the reference's authors published
   (paper_materials/.../LooserSubset_10000_ParCV_5-3-2018.RDS -> tests/golden/published_cv_10000.npz).
 * C restatement (oracle/eben_*.c) against golden vectors produced by the reference's own C.
"""
import math

import numpy as np

from conftest import golden
from oracle import rlayer as R
from oracle.rrng import RRng


def test_rrng_known_answers():
    assert RRng(1, "Rejection").sample_int(10) == [9, 4, 7, 1, 2, 5, 3, 10, 6, 8]    # R >= 3.6.0
    assert RRng(1, "Rounding").sample_int(10) == [3, 4, 5, 7, 2, 8, 9, 6, 10, 1]     # R < 3.6.0
    assert abs(RRng(1).unif_rand() - 0.2655086631421) < 1e-12                         # set.seed(1); runif(1)
    g = golden("rrng.npz")
    assert list(R.assign_to_folds(50, 3)[:12]) == [1, 3, 1, 1, 2, 1, 2, 3, 3, 3, 2, 1]    # SURVEY D.1
    assert list(R.assign_to_folds(500, 5)[:12]) == [4, 2, 4, 3, 1, 4, 5, 1, 2, 2, 1, 5]   # SURVEY D.2
    assert np.array_equal(R.assign_to_folds(1000, 10), g["folds_1000_10"])
    for nf, n in ((3, 50), (5, 500), (10, 1000)):
        f = R.assign_to_folds(n, nf)
        assert np.bincount(f)[1:].max() - np.bincount(f)[1:].min() <= 1


def test_published_cv_table_semantics():
    """Grid values, row order, SE formula and argmin rule against the authors' saved output."""
    p = golden("published_cv_10000.npz")
    alpha = R.r_seq(1.0, 0.05, -0.05)
    assert np.array_equal(np.unique(p["detail_alpha"]), np.sort(alpha))         # bit-for-bit alpha grid
    lam = np.unique(p["detail_lambda"])[::-1]
    lam_max = lam[0]
    lam_min = math.log(0.001 * lam_max)
    mine = np.exp(R.r_seq(math.log(lam_max), lam_min, -(math.log(lam_max) - lam_min) / 19))
    assert np.allclose(mine, lam, rtol=1e-13, atol=0)
    # detail rows: grid-row major (alpha fastest within lambda), fold minor
    assert np.array_equal(p["detail_fold"][:6], [1, 2, 3, 1, 2, 3])
    assert np.allclose(p["detail_alpha"][:9], np.repeat(alpha[:3], 3))
    n_folds = 3
    fold_err = p["detail_mse"].reshape(400, n_folds)
    ga = p["detail_alpha"].reshape(400, n_folds)[:, 0]
    gl = p["detail_lambda"].reshape(400, n_folds)[:, 0]
    s = R.summarise(ga, gl, fold_err)
    assert np.allclose(s["alpha"], p["summary_alpha"]) and np.allclose(s["lambda"], p["summary_lambda"])
    assert np.allclose(s["MSE"], p["summary_mse"], rtol=1e-13)
    assert np.allclose(s["SE"], p["summary_se"], rtol=1e-10)
    a, l, _ = R.select_optimum(s)
    assert a == float(p["alpha_optimal"][0]) and l == float(p["lambda_optimal"][0])


def _port_table(X, y, n_folds, epis, g, kind="port"):
    lib = R.fit_lib(kind)
    out = np.zeros_like(g["fold_err"]); ns = np.zeros_like(g["n_selected"])
    for i, r in enumerate(g["rows"]):
        for f in range(1, n_folds + 1):
            e, fit = R.fit_one(X, y, g["fold_id"], f, g["grid_lambda"][r], g["grid_alpha"][r], epis, "gaussian", lib)
            out[i, f - 1] = e
            ns[i, f - 1] = 0 if fit.weight[0, 0] == 0 else fit.weight.shape[0]
    return out, ns


def test_port_gaussian_config1_matches_reference_golden(bundled, built):
    g = golden("config1_gaussian.npz")
    X, y = bundled["BASIS"][:50, :100].astype(float), bundled["y"][:50]
    ga, gl = R.build_grid(X, y, 3)
    assert np.allclose(ga, g["grid_alpha"], rtol=0, atol=0) and np.allclose(gl, g["grid_lambda"], rtol=1e-14)
    assert abs(gl[0] - 2.5115842672973) < 1e-12 and abs(gl[-1] - 0.0025115842672973) < 1e-15      # SURVEY D.1
    err, ns = _port_table(X, y, 3, False, g)
    assert np.array_equal(ns, g["n_selected"])
    assert np.max(np.abs(err - g["fold_err"]) / np.abs(g["fold_err"])) < 1e-10
    s = R.summarise(ga, gl, err)
    a, l, _ = R.select_optimum(s)
    assert a == 1.0 and abs(l - 0.0222492909371512) < 1e-14                                      # SURVEY D.1
    assert abs(s["MSE"].min() - 1919.181608760305) < 1e-6
    # anchors printed in SURVEY D.1
    assert np.allclose(g["fold_err"][0], [2246.40804244, 2004.15893851, 1558.65730397], rtol=1e-10)
    assert np.allclose(g["fold_err"][399], [2131.74032709, 3156.56558406, 3180.85087744], rtol=1e-10)
    assert list(g["n_selected"][399]) == [9, 8, 9]


def test_port_gaussian_epis_slice(bundled, built):
    g = golden("gauss_epis_slice.npz")
    X, y = bundled["BASIS"][:120, :25].astype(float), bundled["y"][:120]
    err, ns = _port_table(X, y, 3, True, g)
    assert np.array_equal(ns, g["n_selected"])
    assert np.max(np.abs(err - g["fold_err"]) / np.abs(g["fold_err"])) < 1e-10


def test_port_gaussian_bundled_rows(bundled, built):
    g = golden("gauss_bundled_sample.npz")
    X, y = bundled["BASIS"].astype(float), bundled["y"]
    sub = {k: g[k] for k in g.files}
    keep = [0, 3, 9, 17]            # a cheap subset incl. the last (largest active set) row
    sub["rows"] = g["rows"][keep]; sub["fold_err"] = g["fold_err"][keep]; sub["n_selected"] = g["n_selected"][keep]
    err, ns = _port_table(X, y, 3, False, sub)
    assert np.array_equal(ns, sub["n_selected"])
    assert np.max(np.abs(err - sub["fold_err"]) / np.abs(sub["fold_err"])) < 1e-9


def test_local_search_replay_shape_and_rule():
    g = golden("config1_gaussian.npz")
    each, a, l, full = R.local_search_replay(g["grid_alpha"], g["grid_lambda"], g["fold_err"])
    assert each.shape == (20, 4) and full.shape == (400, 4)
    assert np.array_equal(each, g["local_cv"]) and a == float(g["local_alpha"]) and l == float(g["local_lambda"])
    visited = int((full[:, 1] != 0).sum())
    assert 20 <= visited <= 400 and np.all(full[visited:] == 0)
    # first step of every alpha can never stop (previousL = 2e10), so each alpha visits >= 2 lambdas or all
    assert np.all(each[:, 2] <= 1e10)


def test_port_final_model_matches_reference_golden(bundled, built):
    """The whole `.C` output of one fit -- weight table with the posterior variances, intercept, Wald statistic, residual
    variance -- against the reference's own C on config 1 at its optimum (tests/golden/make_golden.py)."""
    g = golden("final_gaussian_config1.npz")
    X, y = bundled["BASIS"][:50, :100].astype(float), bundled["y"][:50]
    f2 = R.eb_elastic_net_gaussian(X, y, float(g["lam"]), float(g["alpha"]), False, R.fit_lib("port"))
    ref = g["raw_beta"]
    assert f2.raw_beta.shape == ref.shape and np.array_equal(f2.raw_beta[:, :2], ref[:, :2])
    assert np.array_equal(f2.raw_beta[:, 2] != 0, ref[:, 2] != 0) and (ref[:, 2] != 0).any()
    assert np.allclose(f2.raw_beta[:, 2:4], ref[:, 2:4], rtol=1e-8, atol=1e-12)
    assert abs(f2.intercept[0] - g["intercept"][0]) < 1e-9 * abs(g["intercept"][0])
    assert abs(f2.wald - float(g["wald"])) <= 1e-8 * max(1.0, abs(float(g["wald"])))
    assert abs(f2.resid_var - float(g["resid_var"])) <= 1e-8 * float(g["resid_var"])


def _port_table_binom(X, y, n_folds, epis, g, rows_idx):
    lib = R.fit_lib("port")
    out = np.zeros((len(rows_idx), n_folds)); ns = np.zeros((len(rows_idx), n_folds), dtype=np.int32)
    for i, ri in enumerate(rows_idx):
        r = g["rows"][ri]
        for f in range(1, n_folds + 1):
            e, fit = R.fit_one(X, y, g["fold_id"], f, g["grid_lambda"][r], g["grid_alpha"][r], epis, "binomial", lib)
            out[i, f - 1] = e
            ns[i, f - 1] = 0 if fit.weight[0, 0] == 0 else fit.weight.shape[0]
    return out, ns


def test_port_binomial_config2_rows(bundled, built):
    """Config 2 (500 x 481 logistic, 5 folds): anchors from SURVEY D.2 and a sample of grid rows."""
    g = golden("config2_binomial.npz")
    X, y = bundled["BASISbinomial"].astype(float), bundled["yBinomial"].astype(float)
    assert abs(g["grid_lambda"][0] - 4.9018946774254) < 1e-12
    assert list(g["fold_id"][:12]) == [4, 2, 4, 3, 1, 4, 5, 1, 2, 2, 1, 5]
    assert abs(float(g["alpha_optimal"]) - 0.2) < 1e-12 and abs(float(g["lambda_optimal"]) - 0.0145897612898799) < 1e-14
    assert abs(g["summary_likelihood"].min() - 0.338311255040) < 1e-10
    assert np.allclose(g["fold_err"][0], [-0.60967424, -0.63577811, -0.62685061, -0.61303727, -0.60829047], atol=1e-8)
    assert np.allclose(g["fold_err"][399], [-0.32703985, -0.28302331, -0.42632759, -0.26404669, -0.42251053], atol=1e-8)
    assert list(g["n_selected"][399]) == [39, 47, 46, 42, 43]
    idx = [0, 45, 130, 399]
    err, ns = _port_table_binom(X, y, 5, False, g, idx)
    assert np.array_equal(ns, g["n_selected"][idx])
    assert np.max(np.abs(err - g["fold_err"][idx]) / np.abs(g["fold_err"][idx])) < 1e-9


def test_port_binomial_epis_slice(bundled, built):
    g = golden("binom_epis_slice.npz")
    X, y = bundled["BASISbinomial"][::4, :20].astype(float), bundled["yBinomial"][::4].astype(float)
    idx = list(range(0, len(g["rows"]), 3))
    err, ns = _port_table_binom(X, y, 3, True, g, idx)
    assert np.array_equal(ns, g["n_selected"][idx])
    ref = g["fold_err"][idx]
    assert np.max(np.abs(err - ref) / np.maximum(np.abs(ref), 1e-12)) < 1e-9


def test_sl_filter_restatement_matches_correlation(bundled):
    """SL_filter.R's statistic |ys' xs| / n is (n-1)/n times the absolute Pearson correlation: check the numpy restatement
    against np.corrcoef on the bundled data (main effects and pairs)."""
    X, y = bundled["BASIS"][:, :30].astype(float), bundled["y"]
    n = X.shape[0]
    main, pairs, sm, sp = R.sl_filter(X, y, 0.05, 0.05)
    assert main.size > 0 and pairs.shape[0] > 0 and np.all(pairs[:, 0] < pairs[:, 1])
    for c, v in zip(main, sm):
        assert abs(v - abs(np.corrcoef(X[:, c - 1], y)[0, 1]) * (n - 1) / n) < 1e-12
    for (i, j), v in list(zip(pairs, sp))[:20]:
        assert abs(v - abs(np.corrcoef(X[:, i - 1] * X[:, j - 1], y)[0, 1]) * (n - 1) / n) < 1e-12
    # every candidate not returned is below its threshold
    allm = np.array([abs(np.corrcoef(X[:, c], y)[0, 1]) * (n - 1) / n for c in range(X.shape[1])])
    assert set(np.nonzero(allm > 0.05)[0] + 1) == set(main.tolist())


def test_sl_filter_restatement_reproduces_reference_held_matrix():
    """oracle/rlayer.py:sl_filter against the kept set of the authors' own filter output (tests/golden/make_sl_golden.py
    verified, where the reference checkout exists, that these are exactly the columns of filter_matrix_main0.05_Zeo)."""
    from conftest import golden
    g = golden("sl_filter_zeo.npz")
    k = int(g["k"])
    X = np.unpackbits(g["bits"], axis=1)[:, :k].astype(np.float64) * 2 - 1
    main, _pairs, stat, _ = R.sl_filter(X, g["y"], float(g["tau_main"]), 0.0, False)
    assert np.array_equal(main - 1, g["kept"]) and np.allclose(stat, g["stat"], rtol=1e-13, atol=0)


def test_streaming_identity(bundled, built):
    """The identity behind the streaming kernels (pareben_b200/csrc/stream.cuh): recomputing S_in / Q_in from the active set
    after every action -- with the beta of the last FullStat and the ghost term of deleted bases -- reproduces the
    reference's incrementally corrected arrays: same supports, results equal far below the 1e-8 parity tolerance."""
    lib = R.fit_lib("port")
    X, y = bundled["BASIS"].astype(float), bundled["y"].astype(float)
    cases = [(X[:300, 100:140], y[:300], True, 0.01, 1.0), (X[:300, 100:140], y[:300], True, 0.02, 0.5),
             (X[:400], y[:400], False, 0.05, 0.5), (X[:400], y[:400], False, 0.02, 1.0)]
    biggest = 0
    try:
        for Xs, ys, epis, lam, al in cases:
            lib.lib.oracle_set_fresh_statistics(0)
            a = R.eb_elastic_net_gaussian(Xs, ys, lam, al, epis, lib)
            lib.lib.oracle_set_fresh_statistics(1)
            b = R.eb_elastic_net_gaussian(Xs, ys, lam, al, epis, lib)
            assert np.array_equal(a.raw_beta[:, 2] != 0, b.raw_beta[:, 2] != 0)
            biggest = max(biggest, a.weight.shape[0])
            assert np.allclose(a.raw_beta[:, 2:4], b.raw_beta[:, 2:4], rtol=1e-9, atol=1e-14)
            assert abs(a.intercept[0] - b.intercept[0]) <= 1e-10 * abs(a.intercept[0]) and abs(a.resid_var - b.resid_var) <= 1e-9 * a.resid_var
    finally:
        lib.lib.oracle_set_fresh_statistics(0)
    assert biggest >= 20                      # the cases do exercise adds, deletes and re-estimates


def test_binomial_irls_accept_reject_depends_on_summation_order(bundled, built):
    """Why binomial parity is stated at 1e-8 and not at rounding level: summing the IRLS data error (NEmainEff.c:2013-2025)
    over the rows in descending instead of ascending order -- the same number up to rounding -- moves some fits of
    config 2 by ~1e-8, because the accept test `newTotalError >= errorLog` (:1991) flips on steps whose true decrease is
    smaller than the rounding of that sum.  Fits whose IRLS steps are all clear-cut do not move at all."""
    from conftest import golden
    g = golden("config2_binomial.npz")
    X, y = bundled["BASISbinomial"].astype(float), bundled["yBinomial"].astype(float)
    P = R.fit_lib("port")
    moved, still = [], []
    try:
        for r, f in ((15, 4), (10, 1), (0, 1), (20, 1)):
            P.lib.oracle_set_reverse_error_sum(0)
            e0, f0 = R.fit_one(X, y, g["fold_id"], f, g["grid_lambda"][r], g["grid_alpha"][r], False, "binomial", P)
            P.lib.oracle_set_reverse_error_sum(1)
            e1, f1 = R.fit_one(X, y, g["fold_id"], f, g["grid_lambda"][r], g["grid_alpha"][r], False, "binomial", P)
            assert f0.weight.shape == f1.weight.shape and abs(e0 - g["fold_err"][r, f - 1]) <= 1e-12 * abs(e0)
            (moved if (r, f) in ((15, 4), (10, 1)) else still).append(abs(e1 - e0) / abs(e0))
    finally:
        P.lib.oracle_set_reverse_error_sum(0)
    assert all(2e-9 < d < 2e-8 for d in moved), moved
    assert all(d < 1e-13 for d in still), still
