"""GPU suite (-m gpu): the binomial score contraction on the int8 tensor cores (tc_contract.cuh).

Binomial main-effect problems whose design holds integers with |x| <= 11 run the FullStat contraction on
tcgen05 int8 MMAs; every other design keeps the FP64 (DMMA) contraction.  Both sides of that choice are
checked fit by fit against the oracle library, on seeded designs with shapes the bundled data does not
reach: training-row counts that are not a multiple of the 32-row stage, candidate counts that are not a
multiple of the 128-candidate tile, an all-zero column, and active sets large enough to need two and three
30-column passes.  Each case also asks the library which contraction ran (pareben_last_contraction_info) and
how many contractions the kernel executed on the tensor cores.  Tolerances as in test_gpu_shapes.py: 5e-8
relative on binomial fold errors, support sizes identical.
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
    return pb


def _contraction(pb, X, y, n_folds, lam, alpha):
    """(tensor-core path chosen, contractions the kernel ran there) for one fit per grid point on fold 1."""
    folds = R.assign_to_folds(X.shape[0], n_folds)
    with pb.Problem(X, y, folds, n_folds, False, "binomial") as p:
        p.run_fits(np.ones(lam.size, np.int32), alpha, lam)
        return p.contraction_info()


def _check(pb, X, y, n_folds, lam, alpha, rtol=5e-8):
    lib = R.fit_lib(R.available_kind())
    folds = R.assign_to_folds(X.shape[0], n_folds)
    err, st, ns = pb.cv_grid(X, y, folds, n_folds, alpha, lam, epis=False, prior="binomial")
    worst, biggest = 0.0, 0
    for i in range(lam.size):
        for f in range(1, n_folds + 1):
            e, fit = R.fit_one(X, y, folds, f, lam[i], alpha[i], False, "binomial", lib)
            m = 0 if fit.weight[0, 0] == 0 else fit.weight.shape[0]
            assert ns[i, f - 1] == m, f"support size differs at lambda={lam[i]}, alpha={alpha[i]}, fold {f}: {ns[i, f - 1]} vs {m}"
            worst = max(worst, abs(err[i, f - 1] - e) / max(abs(e), 1e-300))
            biggest = max(biggest, m)
    assert worst < rtol, f"max relative fold-error difference {worst:.3e}"
    return biggest


def _design(rng, n, k, codes):
    X = rng.choice(codes, size=(n, k)).astype(np.float64)
    for j in range(1, k):                      # linked neighbours, as in genotype data
        keep = rng.random(n) < 0.7
        X[keep, j] = X[keep, j - 1]
    X[:, 5] = 0.0                              # an all-zero candidate
    return X


def _target(rng, X, n_true, size):
    beta = np.zeros(X.shape[1]); beta[rng.choice(np.arange(6, X.shape[1]), n_true, replace=False)] = rng.normal(0, size, n_true)
    eta = (X - X.mean(0)) @ beta
    return (rng.random(X.shape[0]) < 1 / (1 + np.exp(-eta))).astype(np.float64)


def test_codes_012_large_active_sets(pb):
    """{0, 1, 2} codes take the int8 tensor-core path: 283 rows (226 / 227 training rows per fold, not a multiple of
    32), 300 candidates (not a multiple of 128), one all-zero column; small lambdas build active sets past 32 columns."""
    rng = np.random.default_rng(20261020)
    X = _design(rng, 283, 300, [0.0, 1.0, 2.0])
    y = _target(rng, X, 40, 1.2)
    lam = np.array([0.3, 0.02, 0.002, 0.0005]); alpha = np.array([0.9, 0.5, 0.2, 0.05])
    tc, calls = _contraction(pb, X, y, 5, lam, alpha)
    assert tc and calls > 0
    assert _check(pb, X, y, 5, lam, alpha) >= 31


def test_active_set_past_64_columns(pb):
    """Independent {0, 1, 2} loci with many effects: 400 training rows, 300 candidates, active sets past 64 columns,
    so the contraction takes three passes (30 + 30 + the rest)."""
    rng = np.random.default_rng(7)
    n, k, n_true = 600, 300, 150
    X = rng.choice([0.0, 1.0, 2.0], size=(n, k))
    beta = np.zeros(k); beta[rng.choice(k, n_true, replace=False)] = rng.normal(0, 1.5, n_true)
    eta = (X - X.mean(0)) @ beta / np.sqrt(n_true) * 3
    y = (rng.random(n) < 1 / (1 + np.exp(-eta))).astype(np.float64)
    lam = np.array([1e-6]); alpha = np.array([0.01])
    tc, calls = _contraction(pb, X, y, 3, lam, alpha)
    assert tc and calls > 0
    assert _check(pb, X, y, 3, lam, alpha) >= 65


def test_magnitude_12_keeps_the_fp64_contraction(pb):
    """An entry of magnitude 12 (x^2 leaves int8) sends the same kind of design through the DMMA contraction."""
    rng = np.random.default_rng(20261021)
    X = _design(rng, 200, 150, [-1.0, 0.0, 1.0])
    X[7, 9] = 12.0
    X[11, 40] = -12.0
    y = _target(rng, X, 10, 1.0)
    lam = np.array([0.3, 0.03, 0.003]); alpha = np.array([1.0, 0.5, 0.1])
    assert _contraction(pb, X, y, 4, lam, alpha) == (False, 0)
    _check(pb, X, y, 4, lam, alpha)


def test_real_valued_design_keeps_the_fp64_contraction(pb):
    """Non-integer entries: the FP64 contraction, never the tensor cores."""
    rng = np.random.default_rng(20261024)
    X = _design(rng, 180, 140, [-1.0, 0.0, 1.0]) + rng.normal(0, 0.1, (180, 140))
    y = _target(rng, np.round(X), 8, 1.0)
    lam = np.array([0.3, 0.03]); alpha = np.array([1.0, 0.3])
    assert _contraction(pb, X, y, 3, lam, alpha) == (False, 0)
    _check(pb, X, y, 3, lam, alpha)


def test_magnitude_11_small_fold(pb):
    """|x| = 11 is still int8 after squaring: the tensor-core path with large codes and a 61-row training set."""
    rng = np.random.default_rng(20261022)
    X = _design(rng, 92, 130, [-11.0, -3.0, 0.0, 2.0, 11.0])
    y = _target(rng, X, 6, 0.15)
    lam = np.array([0.5, 0.05, 0.005]); alpha = np.array([1.0, 0.6, 0.2])
    tc, calls = _contraction(pb, X, y, 3, lam, alpha)
    assert tc and calls > 0
    _check(pb, X, y, 3, lam, alpha)
