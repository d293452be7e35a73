"""CPU references for the dense linear algebra of a fit (no GPU needed).

tests/test_gpu_linalg_kernels.py holds the kernels of linalg.cuh and contract.cuh to three kinds of reference built here:

* Bit-exact C restatements (tests/kernels/linalg_ref.c, gcc -ffp-contract=off) of the kernels whose arithmetic is plain
  IEEE double in a fixed order: sweep_regs, sweep_core, quad_forms_simt<8>, gram_pipe, cache_dot, sym_matvec_row.
* Inputs whose answer is exact on every path, DMMA included, whose accumulation order is not specified:
  - inverse: A = L D L' with L unit lower bidiagonal (sub-diagonal in {-1, 0, 1}) and D in {1/2, 1, 2}.  The pivots are
    exactly D, and A^-1 = L^-T D^-1 L^-1 has entries that are multiples of 1/2 below 2M.  A pivot D_k <= 0 (or a NaN
    on A's diagonal) is an exactly non-positive pivot at index k.
  - quadratic forms and Gram: small-integer G and PHI, dyadic SIGMA, v and w.
  Exactness in ANY summation order is proved, not assumed: every term is an integer multiple of 2^-s and, for every
  output, the sum of the terms' magnitudes is below 2^(53-s), so every partial sum in any order is representable.  For
  the sweep the terms are those of each rank-1 update, and the sum runs over the pivots of one panel (at most 8), which
  is what the DMMA update sums in an unspecified order (sweep_certificate).
* Accuracy references for realistic inputs (the DMMA paths): the inverse from np.linalg.inv refined once with a
  residual computed in long double (64-bit significand), kept as a double-double; the quadratic forms in long double;
  the Gram matrix exactly (test_contract_reference.exact_dot).  Each is checked against fractions.Fraction at small
  sizes and shown to be at least 2^8 times more accurate than the bound it serves.
"""
import ctypes
import functools
import math
from fractions import Fraction

import numpy as np
import pytest

import kernel_probe as kp
from test_contract_reference import exact_dot

U = 2.0 ** -53
ULD = float(np.finfo(np.longdouble).eps) / 2        # unit roundoff of the reference arithmetic (2^-64 on x86-64)
GRAM_C = 4                                           # bounds: (N + GRAM_C) u ..., (M + QUAD_C) u ..., SWEEP_C M u kappa ...
QUAD_C = 8
SWEEP_C = 2
# the sizes test_gpu_linalg_kernels.py runs the sweep at with the present dispatch constants (it certifies any other)
SWEEP_SIZES = (1, 2, 3, 31, 32, 33, 63, 64, 65, 72, 73, 312, 313, 632, 633, 1024)


@functools.lru_cache(maxsize=None)
def ref_lib():
    L = kp.build_c("linalg_ref")
    d, i = kp.D, ctypes.c_int
    L.ref_sweep_regs.argtypes = [d, i]
    L.ref_sweep_core.argtypes = [d, i]
    L.ref_quad_simt.argtypes = [i, i, d, d, d, d, d]
    L.ref_gram_pipe.argtypes = [i, i, d, d, d, i, d, d]
    L.ref_cache_dot.argtypes = [i, i, d, d, d]
    L.ref_sym_matvec.argtypes = [i, d, d, d]
    return L


# ---------------------------------------------------------------------------------------------------------------------
# the C restatements (column-major matrices as numpy arrays a[j, i] = element (i, j); for symmetric inputs it is moot)

def c_sweep(A, core=False):
    """(ok, a) after ref_sweep_core / ref_sweep_regs on a copy of the M x M matrix A."""
    a = kp.f64(np.array(A, dtype=np.float64, copy=True))
    f = ref_lib().ref_sweep_core if core else ref_lib().ref_sweep_regs
    ok = f(kp.dp(a), a.shape[0])
    return bool(ok), a


def c_quad(G, sigma, v=None):
    """G: logical cache rows [M, Kc]; sigma [M, M] read as sigma[p*M + j]; v [M] or None -> (quad, lin) [Kc]."""
    G = kp.f64(G); M, Kc = G.shape
    q = np.empty(Kc); l = np.empty(Kc)
    ref_lib().ref_quad_simt(M, Kc, kp.dp(G), kp.dp(kp.f64(sigma)), kp.dp(None if v is None else kp.f64(v)), kp.dp(q), kp.dp(l))
    return q, l


def c_gram_pipe(phi, w=None, ev=None, T=256):
    """phi [M, N] -> (H [M, M] with H[j, k] for j <= k and NaN elsewhere, g [M] or None)."""
    phi = kp.f64(phi); M, N = phi.shape
    H = np.full((M, M), np.nan); g = np.full(M, np.nan) if ev is not None else None
    ref_lib().ref_gram_pipe(N, M, kp.dp(phi), kp.dp(None if w is None else kp.f64(w)), kp.dp(None if ev is None else kp.f64(ev)),
                            T, kp.dp(H), kp.dp(g))
    return H, g


def c_cache_dot(G, vec):
    G = kp.f64(G); M, Kc = G.shape
    z = np.empty(Kc)
    ref_lib().ref_cache_dot(M, Kc, kp.dp(G), kp.dp(kp.f64(vec)), kp.dp(z))
    return z


def c_sym_matvec(A, v):
    A = kp.f64(A); M = A.shape[0]
    z = np.empty(M)
    ref_lib().ref_sym_matvec(M, kp.dp(A), kp.dp(kp.f64(v)), kp.dp(z))
    return z


# ---------------------------------------------------------------------------------------------------------------------
# exactness certificates

def grid_exp(x):
    """The smallest s such that every entry of x is an integer multiple of 2^-s (x finite; -inf when all are zero)."""
    x = np.asarray(x, dtype=np.float64).ravel()
    x = x[x != 0]
    if x.size == 0:
        return -math.inf
    m, e = np.frexp(x)
    mi = np.abs(np.ldexp(m, 53)).astype(np.int64)              # exact: |m| in [1/2, 1)
    low = np.log2((mi & -mi).astype(np.float64)).astype(np.int64)
    return int(np.max(53 - low - e))


def sum_certificate(s, mag):
    """True when terms on the 2^-s grid whose magnitudes sum to at most `mag` add up exactly in any order."""
    return bool(np.all(np.asarray(mag) < 2.0 ** (53 - s)))


def sweep_certificate(A, group=8):
    """Prove that the symmetric sweep of A is exact in any summation order within groups of `group` consecutive pivots
    (the panels of sweep_panel; a narrower panel sums a subset).  Simulates the sweep in FP64 -- every operation of which
    the certificate proves exact -- and returns (certified, pivots, -A^-1 as swept).  Only the leading block that the
    pivot column reaches is updated, which makes banded inputs cheap."""
    a = np.array(A, dtype=np.float64, copy=True)
    M = a.shape[0]
    s = grid_exp(a)
    worst = 0.0                                   # largest |entry at group start| + sum of the group's |terms|
    pivots = np.empty(M)
    S = None
    for k in range(M):
        if k % group == 0:
            worst = max(worst, 0.0 if S is None else float(S.max()))
            S = np.abs(a)
        c = a[:, k].copy()
        d = c[k]
        pivots[k] = d
        if not d > 0:
            return False, pivots[:k + 1], a
        m, e = np.frexp(d)
        if m != 0.5:                               # 1/d must be exact: d a power of two
            return False, pivots[:k + 1], a
        dinv = 1.0 / d
        nz = np.nonzero(c)[0]
        n = int(nz[-1]) + 1
        sc = grid_exp(c)
        ed = int(round(math.log2(dinv)))
        s = max(s, 2 * sc - ed, sc - ed, -ed)      # ci*cj*dinv, cj*dinv, dinv
        if np.max(np.abs(c)) ** 2 >= 2.0 ** (53 - 2 * sc):    # ci*cj itself (the FMA form) must be exact
            return False, pivots[:k + 1], a
        T = np.outer(c[:n], c[:n] * dinv)
        S[:n, :n] += np.abs(T)
        a[:n, :n] -= T
        a[k, :] = c * dinv
        a[:, k] = c * dinv
        a[k, k] = -dinv
    worst = max(worst, float(S.max()))
    return sum_certificate(s, worst), pivots, a


def quad_certificate(G, sigma, v=None):
    """quad_c = sum_{j <= p} g_j sigma'_{jp} g_p (sigma' the doubled lower triangle) and lin_c = g'v: exact in any order?"""
    Sd = np.tril(sigma) * 2.0 - np.diag(np.diag(sigma))            # sigma'[p, j] for j <= p (exact)
    # (the grid of sigma itself too: exact_quad_float sums the full symmetric form)
    s = max(grid_exp(G) * 2 + max(grid_exp(Sd), grid_exp(sigma)), grid_exp(G) + (grid_exp(v) if v is not None else -math.inf))
    mag = np.sum(np.abs(G) * (np.abs(Sd) @ np.abs(G)), axis=0)
    ok = sum_certificate(s, mag)
    if v is not None:
        ok = ok and sum_certificate(s, np.abs(v) @ np.abs(G))
    return ok


def gram_certificate(phi, w=None, ev=None):
    """H(j, k) = sum_h fl(phi_j w) phi_k and g = PHI' ev exact in any order (and phi_j w itself exact)?"""
    w = np.ones(phi.shape[1]) if w is None else w
    pw = phi * w
    if grid_exp(pw) > grid_exp(phi) + grid_exp(w) or np.max(np.abs(pw)) >= 2.0 ** (53 - grid_exp(pw)):
        return False
    s = grid_exp(pw) + grid_exp(phi)
    ok = sum_certificate(s, np.abs(pw) @ np.abs(phi).T)
    if ev is not None:
        ok = ok and sum_certificate(grid_exp(phi) + grid_exp(ev), np.abs(phi) @ np.abs(ev))
    return ok


# ---------------------------------------------------------------------------------------------------------------------
# exact cases

def spd_exact(M, seed, fail=None):
    """(A, A^-1, D) for A = L D L' as in the module docstring.  fail = (k, kind) makes pivot k exactly zero, negative or
    NaN (kind 'zero', 'neg', 'nan'); A^-1 is then None."""
    rng = np.random.default_rng([M, seed])
    l = rng.integers(-1, 2, max(M - 1, 0)).astype(np.float64)
    D = np.ldexp(1.0, rng.integers(-1, 2, M))
    if fail is not None:
        k, kind = fail
        D[k] = {"zero": 0.0, "neg": -1.0, "nan": 1.0}[kind]
    L = np.eye(M) + np.diag(l, -1)
    A = (L * D) @ L.T                                             # entries l^2 D + D and l D: exact
    if fail is not None:
        if fail[1] == "nan":
            A[fail[0], fail[0]] = np.nan
        return A, None, D
    Linv = np.eye(M)                                              # (L^-1)[i, j] = prod_{j <= m < i} (-l_m)
    for j in range(M - 1):
        Linv[j + 1:, j] = np.cumprod(-l[j:])
    terms = Linv / D[:, None]
    assert sum_certificate(1, np.abs(Linv).T @ np.abs(terms))    # multiples of 1/2: A^-1 below is exact
    Ainv = Linv.T @ terms
    return A, Ainv, D


def int_cache(rng, M, Kc, lo=-3, hi=3):
    return rng.integers(lo, hi + 1, (M, Kc)).astype(np.float64)


def dyadic(rng, shape, s=4, lim=2.0):
    return np.round(rng.uniform(-lim, lim, shape) * 2.0 ** s) / 2.0 ** s


def dyadic_sym(rng, M, s=4, lim=2.0):
    S = dyadic(rng, (M, M), s, lim)
    return np.tril(S) + np.tril(S, -1).T


def exact_quad(G, sigma, v=None):
    """The exact quad (and lin) of integer G and dyadic symmetric sigma, in Python integers."""
    s = max(0, grid_exp(sigma), grid_exp(v) if v is not None else 0)
    Si = (sigma * 2.0 ** s).astype(np.int64).astype(object)
    Gi = G.astype(np.int64).astype(object)
    q = np.array([float(Fraction(int(x), 2 ** s)) for x in np.sum(Gi * Si.dot(Gi), axis=0)])
    if v is None:
        return q, np.zeros(G.shape[1])
    vi = (v * 2.0 ** s).astype(np.int64).astype(object)
    return q, np.array([float(Fraction(int(x), 2 ** s)) for x in vi.dot(Gi)])


def exact_quad_float(G, sigma, v=None):
    """quad and lin in FP64: the exact values for inputs quad_certificate accepts (every partial sum is exact)."""
    return np.sum(G * (sigma @ G), axis=0), (v @ G if v is not None else np.zeros(G.shape[1]))


# ---------------------------------------------------------------------------------------------------------------------
# realistic inputs and accuracy references

def hessian(rng, N, M, alpha_range=(1e-3, 1e6)):
    """(PHI [M, N], w [N], H = PHI' B PHI + diag(0, alpha)) as a binomial fit forms them: column 0 the intercept, the
    others normalised genotype columns (codes 0/1/2), sigmoid weights clamped as post_mode clamps them, and alpha
    log-uniform over alpha_range."""
    maf = rng.uniform(0.05, 0.5, M - 1)
    X = rng.binomial(2, maf, (N, M - 1)).astype(np.float64)
    X[0, X.sum(axis=0) == 0] = 1.0
    phi = np.vstack([np.ones(N), (X / np.sqrt((X * X).sum(axis=0))).T])
    eta = rng.normal(0, 2.5, N)
    eta[: max(1, N // 50)] = rng.choice([-40.0, 40.0], max(1, N // 50))          # saturated rows: the 1e-10 clamp
    y = 1.0 / (1.0 + np.exp(-eta))
    w = y * (1 - y)
    w[w < 1e-10] = 1e-5
    w[w > 1e10] = 1e5
    alpha = np.exp(rng.uniform(np.log(alpha_range[0]), np.log(alpha_range[1]), M - 1))
    H = (phi * w) @ phi.T
    H = np.triu(H) + np.triu(H, 1).T                                              # exactly symmetric
    H[np.arange(1, M), np.arange(1, M)] += alpha
    return phi, w, H


def pow2_scaling(A):
    """e with S = diag(2^e) making the diagonal of S A S lie in [1/2, 2): the sweep of S A S is exactly S^-1 (sweep of A)
    S^-1 (scaling by powers of two changes no rounding; test_gpu_linalg_kernels checks it bitwise), so the error of an
    inverse can be measured in that frame, where kappa is near its minimum over diagonal scalings (van der Sluis)."""
    return -np.round(np.log2(np.diag(A)) / 2).astype(np.int64)


def scale2(A, e):
    return np.ldexp(np.ldexp(A, e[:, None]), e[None, :])


def inverse_ref(A):
    """A^-1 in the frame of pow2_scaling, as a double-double (X0, C) of S^-1 A^-1 S^-1: X0 = np.linalg.inv(S A S),
    C = X0 (I - S A S X0) with the residual in long double."""
    As = scale2(A, pow2_scaling(A))
    X0 = np.linalg.inv(As)
    X0 = (X0 + X0.T) / 2
    Al, Xl = As.astype(np.longdouble), X0.astype(np.longdouble)
    R = np.eye(A.shape[0], dtype=np.longdouble) - Al @ Xl
    C = (Xl @ R).astype(np.float64)
    return X0, C


def inverse_bound(A):
    """SWEEP_C M u kappa_2(S A S) ||(S A S)^-1||_2 (see test_gpu_linalg_kernels.py), the bound on the error of an inverse
    in the frame of pow2_scaling, and ||(S A S)^-1||_2."""
    ev = np.linalg.eigvalsh(scale2(A, pow2_scaling(A)))
    M = A.shape[0]
    return SWEEP_C * M * U * (ev[-1] / ev[0]) / ev[0], 1.0 / ev[0]


def inverse_err(X, A, ref):
    """||S^-1 X S^-1 - (S A S)^-1||_2 for a computed inverse X of A (S from pow2_scaling, ref = inverse_ref(A))."""
    X0, C = ref
    Xs = scale2(X, -pow2_scaling(A))
    return np.linalg.norm((Xs - X0) - C, 2)


def quad_ref(G, sigma, v=None):
    """quad and lin in long double (sigma symmetric)."""
    Gl = G.astype(np.longdouble)
    q = np.sum(Gl * (sigma.astype(np.longdouble) @ Gl), axis=0)
    l = (v.astype(np.longdouble) @ Gl) if v is not None else np.zeros(G.shape[1], np.longdouble)
    return q, l


def quad_bound(G, sigma, v=None):
    M = G.shape[0]
    qb = (M + QUAD_C) * U * np.sum(np.abs(G) * (np.abs(sigma) @ np.abs(G)), axis=0)
    lb = (M + QUAD_C) * U * (np.abs(v) @ np.abs(G)) if v is not None else np.zeros(G.shape[1])
    return qb, lb


def gram_ref(phi, w):
    """Exact sum_h fl(phi_j w) phi_k as (hi, lo) [M, M]."""
    pw = phi * w
    hi, lo = exact_dot(pw.T, phi.T)
    return hi.T, lo.T


def gram_bound(phi, w):
    N = phi.shape[1]
    return (N + GRAM_C) * U * (np.abs(phi * w) @ np.abs(phi).T)


def ratio(err, bound):
    err = np.asarray(err, dtype=np.float64); bound = np.asarray(bound, dtype=np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        r = np.where(err == 0, 0.0, err / bound)
    return float(np.max(r)) if r.size else 0.0


# ---------------------------------------------------------------------------------------------------------------------
# tests: the references themselves

def _frac_inv(A):
    M = A.shape[0]
    a = [[Fraction(float(A[i, j])) for j in range(M)] + [Fraction(int(i == j)) for j in range(M)] for i in range(M)]
    for k in range(M):
        p = a[k][k]
        a[k] = [x / p for x in a[k]]
        for i in range(M):
            if i != k and a[i][k] != 0:
                f = a[i][k]
                a[i] = [x - f * y for x, y in zip(a[i], a[k])]
    return [[a[i][M + j] for j in range(M)] for i in range(M)]


@pytest.mark.parametrize("M", SWEEP_SIZES)
def test_exact_inverse_family_is_certified(M):
    """Every exact inverse case the GPU test uses is exact in any order within a panel, and its pivots are D."""
    A, Ainv, D = spd_exact(M, 0)
    ok, piv, a = sweep_certificate(A)
    assert ok, f"M={M}: sweep not certified exact"
    assert np.array_equal(piv, D)
    assert np.array_equal(-a, Ainv)
    if M <= 12:
        F = _frac_inv(A)
        assert all(Fraction(float(Ainv[i, j])) == F[i][j] for i in range(M) for j in range(M))


def test_certificates_reject_inexact_inputs():
    A, _, _ = spd_exact(40, 1)
    A[0, 0] = 3.0                                                  # a pivot that is not a power of two
    assert not sweep_certificate(A)[0]
    rng = np.random.default_rng(5)
    G = int_cache(rng, 20, 30)
    assert not quad_certificate(G, rng.normal(size=(20, 20)))
    assert not gram_certificate(int_cache(rng, 8, 40), rng.uniform(0.1, 0.2, 40))


@pytest.mark.parametrize("M,core", [(1, False), (5, False), (32, False), (33, False), (64, False), (1, True), (40, True), (100, True)])
def test_c_sweep_exact(M, core):
    A, Ainv, _ = spd_exact(M, 2)
    assert sweep_certificate(A)[0]
    ok, X = c_sweep(A, core)
    assert ok and np.array_equal(X, Ainv)


@pytest.mark.parametrize("core", [False, True])
@pytest.mark.parametrize("kind", ["zero", "neg", "nan"])
def test_c_sweep_failure(core, kind):
    for k in (0, 7, 19):
        A, _, _ = spd_exact(20, 3, (k, kind))
        assert not c_sweep(A, core)[0]


@pytest.mark.parametrize("M", [3, 24, 64])
def test_c_sweep_realistic_within_bound(M):
    rng = np.random.default_rng(M)
    _, _, A = hessian(rng, 2 * M + 10, M)
    ref = inverse_ref(A)
    bound, _ = inverse_bound(A)
    for core in (False, True):
        ok, X = c_sweep(A, core)
        assert ok and np.array_equal(X, X.T)
        r = inverse_err(X, A, ref) / bound
        assert r <= 1.0, f"sweep_{'core' if core else 'regs'} M={M}: error/bound {r:.3g}"


@pytest.mark.parametrize("M", [2, 4, 7])
def test_inverse_reference_against_fractions(M):
    """The refined inverse is at least 2^8 times more accurate than the bound it serves."""
    rng = np.random.default_rng(100 + M)
    _, _, A = hessian(rng, 12, M, (1e-2, 1e3))
    X0, C = inverse_ref(A)
    e = pow2_scaling(A)
    F = _frac_inv(A)
    err = max(abs(Fraction(float(X0[i, j])) + Fraction(float(C[i, j])) - F[i][j] / Fraction(2) ** int(e[i] + e[j]))
              for i in range(M) for j in range(M))
    bound, _ = inverse_bound(A)
    # ||E||_2 <= M max|E_ij|
    assert M * float(err) * 2 ** 8 <= bound, f"M={M}: reference error {float(err):.3g}, bound {bound:.3g}"


@pytest.mark.parametrize("M,Kc", [(1, 1), (3, 7), (8, 9), (9, 33), (31, 40), (64, 129)])
def test_c_quad_exact(M, Kc):
    rng = np.random.default_rng(M * 1000 + Kc)
    G = int_cache(rng, M, Kc); S = dyadic_sym(rng, M); v = dyadic(rng, M)
    assert quad_certificate(G, S, v)
    q, l = c_quad(G, S, v)
    eq, el = exact_quad(G, S, v)
    assert np.array_equal(q, eq) and np.array_equal(l, el)
    fq, fl = exact_quad_float(G, S, v)
    assert np.array_equal(fq, eq) and np.array_equal(fl, el)


@pytest.mark.parametrize("M", [3, 8, 17])
def test_quad_reference_against_fractions(M):
    rng = np.random.default_rng(M)
    G = rng.normal(size=(M, 5)); S = rng.normal(size=(M, M)); S = (S + S.T) / 2; v = rng.normal(size=M)
    q, l = quad_ref(G, S, v)
    qb, lb = quad_bound(G, S, v)
    for c in range(5):
        g = [Fraction(float(x)) for x in G[:, c]]
        eq = sum(g[i] * Fraction(float(S[i, j])) * g[j] for i in range(M) for j in range(M))
        el = sum(g[i] * Fraction(float(v[i])) for i in range(M))
        assert abs(Fraction(*q[c].as_integer_ratio()) - eq) * 2 ** 8 <= Fraction(float(qb[c]))
        assert abs(Fraction(*l[c].as_integer_ratio()) - el) * 2 ** 8 <= Fraction(float(lb[c]))


@pytest.mark.parametrize("M", [2, 40, 64])
def test_c_quad_realistic_within_bound(M):
    rng = np.random.default_rng(7 + M)
    _, _, H = hessian(rng, 3 * M, M)
    S = np.linalg.inv(H); S = (S + S.T) / 2
    G = rng.normal(size=(M, 50)); v = rng.normal(size=M)
    q, l = c_quad(G, S, v)
    rq, rl = quad_ref(G, S, v)
    qb, lb = quad_bound(G, S, v)
    assert ratio(np.abs(q - rq).astype(np.float64), qb) <= 1 and ratio(np.abs(l - rl).astype(np.float64), lb) <= 1


@pytest.mark.parametrize("N,M", [(1, 1), (2, 5), (33, 4), (64, 32), (65, 33), (130, 64), (1001, 17)])
def test_c_gram_pipe_exact(N, M):
    rng = np.random.default_rng(N * 100 + M)
    phi = int_cache(rng, M, N, -2, 2); w = np.ldexp(rng.integers(1, 17, N).astype(np.float64), -6); ev = dyadic(rng, N)
    assert gram_certificate(phi, w, ev)
    H, g = c_gram_pipe(phi, w, ev)
    E = (phi * w) @ phi.T                                          # exact (certified)
    iu = np.triu_indices(M)
    assert np.array_equal(H[iu], E[iu]) and np.array_equal(g, phi @ ev)


@pytest.mark.parametrize("N,M", [(7, 3), (40, 20)])
def test_gram_reference_against_fractions(N, M):
    rng = np.random.default_rng(N + M)
    phi, w, _ = hessian(rng, N, M)
    hi, lo = gram_ref(phi, w)
    pw = phi * w
    for j in range(M):
        for k in range(j, M):
            e = sum(Fraction(float(pw[j, h])) * Fraction(float(phi[k, h])) for h in range(N))
            assert Fraction(float(hi[j, k])) + Fraction(float(lo[j, k])) - e == 0 or \
                abs(Fraction(float(hi[j, k])) + Fraction(float(lo[j, k])) - e) <= abs(e) * Fraction(2) ** -100


@pytest.mark.parametrize("N,M", [(50, 8), (500, 40), (333, 64)])
def test_c_gram_pipe_realistic_within_bound(N, M):
    rng = np.random.default_rng(N + 3 * M)
    phi, w, _ = hessian(rng, N, M)
    H, _ = c_gram_pipe(phi, w)
    hi, lo = gram_ref(phi, w)
    iu = np.triu_indices(M)
    assert ratio(np.abs((H - hi) - lo)[iu], gram_bound(phi, w)[iu]) <= 1


def test_c_cache_dot_and_sym_matvec():
    rng = np.random.default_rng(11)
    for M in (1, 3, 4, 5, 8, 33):
        G = int_cache(rng, M, 21); vec = dyadic(rng, M)
        assert np.array_equal(c_cache_dot(G, vec), G.T @ vec)      # small integers times dyadics: exact
        A = dyadic_sym(rng, M)
        assert np.array_equal(c_sym_matvec(A, vec), A @ vec)
        # the chains: an order that differs from (z0 + z1) + (z2 + z3) is visible with cancelling terms
    A = np.zeros((5, 5)); A[0, 0] = 1.0; A[1, 0] = 2.0 ** 53; A[2, 0] = 1.0; A[3, 0] = -(2.0 ** 53)
    z = c_sym_matvec(A, np.ones(5))
    assert z[0] == ((1.0 + 2.0 ** 53) + (1.0 - 2.0 ** 53))
