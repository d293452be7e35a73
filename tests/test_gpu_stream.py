"""GPU suite (-m gpu), part 3: the streaming-Kc mode (pareben_b200/csrc/stream*.cuh).

Streaming mode keeps no per-candidate array: the statistics the reference maintains incrementally (S_in, Q_in of
elasticNetLinearNeFull2.c:1063-1196 and the action corrections) are recomputed every inner iteration by one dense
contraction per fold for all fits at once.  It is what BASELINE config 5 (Kc = 2e8) needs; here it is forced
(pareben_set_mode(2)) on problems small enough for the CPU oracle and compared fit by fit with oracle/_ref (or the C
restatement), and with the cached kernel's table.  Tolerance: 1e-8 relative on fold errors, identical supports.
"""
import numpy as np
import pytest

from oracle import rlayer as R

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pb(built):
    import pareben_b200 as pb
    if pb.device_count() < 1:
        pytest.fail("no CUDA device: the -m gpu suite must run on the B200 box")
    yield pb
    pb.set_mode(pb.MODE_AUTO)


def _genotypes(rng, n, k, block=25, copy=0.85):
    X = rng.choice([-1.0, 0.0, 1.0], size=(n, k), p=[0.25, 0.5, 0.25])
    for j in range(1, k):
        if j % block:
            keep = rng.random(n) < copy
            X[keep, j] = X[keep, j - 1]
    return X


def _stream_vs_oracle(pb, X, y, n_folds, lam, alpha, epis, rtol=1e-8, check_folds=None):
    folds = R.assign_to_folds(X.shape[0], n_folds)
    pb.set_mode(pb.MODE_STREAMING)
    try:
        with pb.Problem(X, y, folds, n_folds, epis=epis) as prob:
            assert prob.streaming
            err, st, ns = prob.cv_grid(alpha, lam)
            scan_ms, scan_flops, scans, rounds = prob.stream_counters()
    finally:
        pb.set_mode(pb.MODE_AUTO)
    assert scans > 0 and rounds > 0 and scan_flops > 0
    assert np.all(st == 0), st
    lib = R.fit_lib(R.available_kind())
    worst, biggest = 0.0, 0
    for i in range(lam.size):
        for f in (check_folds or range(1, n_folds + 1)):
            e, fit = R.fit_one(X, y, folds, f, lam[i], alpha[i], epis, "gaussian", lib)
            m = 0 if fit.weight[0, 0] == 0 else fit.weight.shape[0]
            assert ns[i, f - 1] == m, f"support differs at lambda={lam[i]}, alpha={alpha[i]}, fold {f}: {ns[i, f - 1]} vs {m}"
            worst = max(worst, abs(err[i, f - 1] - e) / max(abs(e), 1e-300))
            biggest = max(biggest, m)
    assert worst < rtol, f"max relative fold-error difference {worst:.3e}"
    return err, biggest


def test_stream_config1_slice_matches_oracle_and_cached(pb):
    """Config 1's data (bundled BASIS[1:50,1:100]) through both organisations of the solver."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "inputs_bundled.npz"))
    X = g["BASIS"][:50, :100].astype(np.float64); y = g["y"][:50]
    grid = pb.BuildGrid(X, y, 3)
    rows = np.arange(0, 400, 13)
    lam, alpha = grid["lambda"][rows], grid["alpha"][rows]
    err_s, _ = _stream_vs_oracle(pb, X, y, 3, lam, alpha, False)
    folds = R.assign_to_folds(50, 3)
    err_c, st, _ = pb.cv_grid(X, y, folds, 3, alpha, lam)
    assert np.max(np.abs(err_s - err_c) / np.abs(err_c)) < 1e-9


def test_stream_epis_gaussian_pairs(pb):
    """Epis: 60 loci -> 1,830 candidates, pair columns generated in registers; active sets of a few dozen."""
    rng = np.random.default_rng(7)
    n, k = 200, 60
    X = _genotypes(rng, n, k, block=10)
    y = 50 + 2.5 * X[:, 3] - 2.0 * X[:, 40] + 3.0 * X[:, 7] * X[:, 22] - 2.5 * X[:, 31] * X[:, 55] + rng.normal(0, 2.0, n)
    lam = np.array([1.5, 0.4, 0.1, 0.03]); alpha = np.array([1.0, 0.5, 0.1, 0.7])
    _, m = _stream_vs_oracle(pb, X, y, 3, lam, alpha, True)
    assert m >= 4


def test_stream_main_effects_bundled_rows(pb):
    """Bundled 481-marker design, 300 rows: active sets up to ~100 with deletes and re-estimates."""
    import os
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "inputs_bundled.npz"))
    X = g["BASIS"][:300].astype(np.float64); y = g["y"][:300]
    lam = np.array([0.6, 0.15, 0.05, 0.02]); alpha = np.array([1.0, 0.5, 0.2, 0.05])
    _, m = _stream_vs_oracle(pb, X, y, 3, lam, alpha, False)
    assert m >= 30


def test_stream_real_valued_design(pb):
    """Non-genotype design: the f64 operand path of the scan (no int8 copy exists); main effects, then pairs."""
    rng = np.random.default_rng(12)
    n, k = 150, 60
    X = rng.normal(size=(n, k))
    X[:, 10] = 0.6 * X[:, 3] + 0.8 * X[:, 10]                 # some collinearity
    y = 10 + X[:, :6] @ np.array([2.0, -1.5, 1.0, 0.8, -0.6, 0.5]) + rng.normal(0, 1.0, n)
    _stream_vs_oracle(pb, X, y, 3, np.array([1.0, 0.2, 0.04]), np.array([1.0, 0.5, 0.1]), False)
    _stream_vs_oracle(pb, X[:, :14], y, 2, np.array([0.8, 0.1]), np.array([0.9, 0.2]), True)


def test_stream_many_fits_many_tiles(pb):
    """More waiting fits than one 64-wide right-hand-side tile per fold, on a 300-locus design made with the config-5
    recipe (45,150 candidates): the streamed table must equal the cached kernel's to rounding and be reproducible."""
    rng = np.random.default_rng(20260101)
    n, k = 600, 300
    X = _genotypes(rng, n, k, block=50, copy=0.9)
    beta = np.zeros(k); beta[rng.choice(k, 6, replace=False)] = rng.normal(0, 2.0, 6)
    pairs = rng.choice(k, (4, 2), replace=False)
    y = 100 + X @ beta + sum(rng.normal(0, 2.0) * X[:, a] * X[:, b] for a, b in pairs) + rng.normal(0, 3.0, n)
    folds = R.assign_to_folds(n, 2)
    grid = pb.BuildGrid(X, y, 2, Epis="yes")
    rows = np.arange(0, 400, 3)                       # 134 grid points x 2 folds: 67 per fold -> two tiles per fold
    lam, alpha = grid["lambda"][rows], grid["alpha"][rows]
    pb.set_mode(pb.MODE_STREAMING)
    try:
        err_a, st_a, ns_a = pb.cv_grid(X, y, folds, 2, alpha, lam, epis=True)
        err_b, st_b, ns_b = pb.cv_grid(X, y, folds, 2, alpha, lam, epis=True)
    finally:
        pb.set_mode(pb.MODE_AUTO)
    assert np.array_equal(err_a, err_b) and np.array_equal(ns_a, ns_b)      # schedule-independent
    err_c, st_c, ns_c = pb.cv_grid(X, y, folds, 2, alpha, lam, epis=True)
    assert np.array_equal(ns_a, ns_c)
    assert np.max(np.abs(err_a - err_c) / np.abs(err_c)) < 1e-8


def test_stream_k2000_slice_against_reference_fixture(pb):
    """K = 2,000 loci of the config-5 recipe, Epis = "yes": 2,001,000 candidates, the golden values of
    tests/golden/make_stream_golden.py (the reference's own C).  Rows of BuildGrid's own grid keep one basis (the
    regime of config 5 at full size); lambda = 0.07 builds ~110 effects out of two million candidates."""
    from conftest import golden
    from pareben_b200.synth import config5
    g = golden("stream_k2000.npz")
    d = config5(int(g["n"]), int(g["k"]), int(g["seed"]))
    X = d["X"].astype(np.float64); y = d["y"]
    assert np.array_equal(y[:8], g["y_check"])                       # the generator reproduces the fixture's data
    nf = int(g["n_folds"])
    folds = g["fold_id"]
    have = np.isfinite(g["fold_err"])
    gi, fi = np.nonzero(have)
    assert abs(pb.GetLambdaMax(X, y, "yes") - float(g["lambda_max"])) <= 1e-12 * float(g["lambda_max"])
    pb.set_mode(pb.MODE_STREAMING)
    try:
        with pb.Problem(X, y, folds, nf, epis=True) as prob:
            assert prob.streaming
            err, st, ns, it = prob.run_fits(fi + 1, g["alpha"][gi], g["lam"][gi])
    finally:
        pb.set_mode(pb.MODE_AUTO)
    assert np.all(st == 0)
    want_e, want_m = g["fold_err"][gi, fi], g["n_selected"][gi, fi]
    assert np.array_equal(ns, want_m), (ns, want_m)
    assert ns.max() >= 100
    rel = np.abs(err - want_e) / np.abs(want_e)
    assert rel.max() < 1e-8, rel

