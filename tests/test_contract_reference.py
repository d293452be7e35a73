"""CPU references for the score contractions (no GPU needed).

Two references that tests/test_gpu_contract_kernels.py holds the kernels to:

* exact_dot: the exact value of X'B for double-valued X and B.  Every double is a dyadic rational, so each column is
  cut into integer limbs of a few bits (V = sum_k L_k 2^(E - b(k+1)), exact), the limbs are multiplied with float64
  matrix products whose sums stay below 2^53 (exact), and the limb products are recombined in Python integers.  The
  result comes back as a double-double (hi, lo): hi is the correctly rounded value, lo the rest.
* tc_emulate: a bit-exact numpy restatement of tc_contract (tc_contract.cuh): the column scaling, the 56-bit fixed
  point, the balanced base-128 digits exactly as tc_digits peels them off, exact per-plane integer sums, Horner in FP64,
  the scale, and div_by with its two FMAs evaluated exactly.

The tests here check both references: exact_dot against fractions.Fraction, the digits against the integers they
encode, and the emulation against exact_dot within the bound the kernel documents, N 2^-57 max|b| max|x|.
"""
import math
from fractions import Fraction

import numpy as np
import pytest

DBL_MAX = np.finfo(np.float64).max
TC_BOUND = 2.0 ** -57          # tc_contract: |error| <= N 2^-57 max|b| max|x| before the division by the column norm


# ---------------------------------------------------------------------------------------------------------------------
# exact X'B

def _limbs(V, bits):
    """V [N, m] doubles -> (L [n, N, m] integer-valued doubles with |L| < 2^bits, E [m]) such that, exactly,
    V[:, j] = sum_k L[k, :, j] 2^(E[j] - bits (k + 1))."""
    V = np.asarray(V, dtype=np.float64)
    _, E = np.frexp(np.abs(V).max(axis=0))            # |V[:, j]| < 2^E[j]
    E = E.astype(np.int64)
    U = np.ldexp(V, -E[None, :])
    assert np.array_equal(np.ldexp(U, E[None, :]), V), "column spans too many binades for an exact scaling"
    out = []
    while np.any(U != 0):
        U = U * 2.0 ** bits
        D = np.trunc(U)
        U = U - D
        out.append(D)
    if not out:
        out.append(np.zeros_like(V))
    return np.array(out), E


def exact_dot(A, B):
    """Exact A'B for A [N, Kc], B [N, R] (finite doubles) as a double-double (hi, lo), each [R, Kc]."""
    A = np.asarray(A, dtype=np.float64)
    B = np.asarray(B, dtype=np.float64)
    N = A.shape[0]
    nbits = max(1, math.ceil(math.log2(N + 1)))
    a_int = bool(np.all(A == np.trunc(A))) and np.abs(A).max() < 2.0 ** 15
    if a_int:                                          # one limb: the integers themselves
        ab = max(1, math.ceil(math.log2(np.abs(A).max() + 1)))
        La, Ea = A[None], np.full(A.shape[1], ab, np.int64)
    else:
        ab = (53 - nbits) // 2
        La, Ea = _limbs(A, ab)
    bb = 53 - nbits - ab
    assert bb >= 8
    Lb, Eb = _limbs(B, bb)
    na, nb = La.shape[0], Lb.shape[0]
    acc = np.zeros((A.shape[1], B.shape[1]), dtype=object)
    for i in range(na):
        for k in range(nb):
            S = La[i].T @ Lb[k]                        # every partial sum is an integer below 2^53: exact
            shift = (na - 1 - i) * ab + (nb - 1 - k) * bb
            acc += S.astype(np.int64).astype(object) * (1 << shift)
    base = Ea[:, None] + Eb[None, :] - na * ab - nb * bb
    hi = np.empty(acc.shape)
    lo = np.empty(acc.shape)
    for idx in np.ndindex(acc.shape):
        v = Fraction(int(acc[idx])) * Fraction(2) ** int(base[idx])
        hi[idx] = float(v)
        lo[idx] = float(v - Fraction(hi[idx]))
    return hi.T, lo.T


def abs_dot(A, B):
    """sum_h |a_h| |b_h| in FP64 ([R, Kc]): only a bound is built from it."""
    return (np.abs(np.asarray(B, np.float64)).T @ np.abs(np.asarray(A, np.float64)))


def err_vs(got, hi, lo, scale=None):
    """|got - exact| (exact = hi + lo, divided by `scale` per candidate when given), in FP64."""
    if scale is None:
        return np.abs((got - hi) - lo)
    q = np.array([[float((Fraction(h) + Fraction(l)) / Fraction(s)) for h, l, s in zip(hr, lr, scale)] for hr, lr in zip(np.atleast_2d(hi), np.atleast_2d(lo))])
    return np.abs(np.atleast_2d(got) - q).reshape(np.shape(got))


# ---------------------------------------------------------------------------------------------------------------------
# tc_contract, bit for bit

def tc_digits(q):
    """Balanced base-128 digits of q (int64, |q| < 2^55), least significant plane last: D [8, ...] with q =
    sum_s D[s] 128^(7-s), as tc_digits extracts them (low 28 bits give planes 7..4 and a carry, the rest planes 3..0)."""
    q = np.asarray(q, dtype=np.int64)
    lo = q & 0xfffffff
    hi = q >> 28
    D = np.zeros((8,) + q.shape, dtype=np.int64)
    for s in range(7, -1, -1):
        x = lo if s >= 4 else hi
        d = ((x + 64) & 127) - 64
        x = (x - d) >> 7
        if s >= 4:
            lo = x
        else:
            hi = x
        if s == 4:
            hi = hi + lo
        D[s] = d + (x << 7) if s == 0 else d
    return D


def tc_column(v):
    """The per-column set-up of tc_digits for one right-hand-side column v [N]:
    (q [N] int64, scale applied after Horner's sum, bad).  The column's scale 2^(ex+1) is stored as 2^(ex-1), and Horner's
    last step multiplies by 2^-5 instead of 2^-7 (2^(ex+1) itself overflows for a column maximum >= 2^1022)."""
    a = np.abs(v)
    bad = not np.all(a <= DBL_MAX)
    mx = 0.0 if bad else float(a.max()) if a.size else 0.0
    _, ex = math.frexp(mx)
    live = not bad and mx > 1e-290
    if not live:
        return np.zeros(v.shape, np.int64), (math.nan if bad else 0.0), bad
    q = np.rint(v * math.ldexp(1.0, 55 - ex)).astype(np.int64)
    return q, math.ldexp(1.0, ex - 1), bad


def fma_exact(a, b, c):
    """Correctly rounded a*b + c, elementwise."""
    a, b, c = np.broadcast_arrays(np.asarray(a, np.float64), np.asarray(b, np.float64), np.asarray(c, np.float64))
    out = np.empty(a.shape)
    for idx in np.ndindex(a.shape):
        x, y, z = float(a[idx]), float(b[idx]), float(c[idx])
        if math.isfinite(x) and math.isfinite(y) and math.isfinite(z):
            v = Fraction(x) * Fraction(y) + Fraction(z)
            try:
                out[idx] = float(v)
            except OverflowError:
                out[idx] = math.inf if v > 0 else -math.inf
        else:
            out[idx] = x * y + z
    return out


def div_by(a, b):
    """gauss_fit.cuh div_by(a, b, 1/b): q = a r, then fma(fma(-q, b, a), r, q)."""
    r = 1.0 / b
    q = a * r
    return fma_exact(fma_exact(-q, b, a), r, q)


def tc_emulate(X, phi, w, e, scale=None, return_planes=False):
    """tc_contract on X [N, K] (integers), phi [R, N], w [N], e [N]: (G [R, K], bb [K], ze [K]).
    G is divided by `scale` [K] with div_by when it is given, else returned before the division."""
    X = np.asarray(X, dtype=np.float64)
    N, K = X.shape
    phi = np.asarray(phi, dtype=np.float64).reshape(-1, N)
    R = phi.shape[0]
    with np.errstate(invalid="ignore", over="ignore"):
        V = np.concatenate([w[None, :] * phi, np.asarray(e, np.float64)[None, :]], axis=0)     # [R + 1, N], FP64
    Q = np.zeros(V.shape, np.int64)
    bscale = np.zeros(R + 1)
    for j in range(R + 1):
        Q[j], bscale[j], _ = tc_column(V[j])
    D = tc_digits(Q)                                                   # [8, R + 1, N]
    # plane sums [8, R + 1, K] and X o X against column 0's planes: integers below 2^31, so FP64 products are exact
    Df = D.astype(np.float64)
    acc = np.stack([Df[s] @ X for s in range(8)]).astype(np.int64)
    acc_bb = np.stack([Df[s, 0] @ (X * X) for s in range(8)]).astype(np.int64)
    with np.errstate(invalid="ignore", over="ignore"):
        v = np.zeros((R + 1, K))
        vb = np.zeros(K)
        for s in range(7, -1, -1):
            v = (v + acc[s].astype(np.float64)) * (0.0078125 if s else 0.03125)
            vb = (vb + acc_bb[s].astype(np.float64)) * (0.0078125 if s else 0.03125)
        v = v * bscale[:, None]
        vb = vb * bscale[0]
    G = v[:R]
    if scale is not None and R > 0:
        G = np.stack([div_by(G[j], np.asarray(scale, np.float64)) for j in range(R)])
    out = (G, vb, v[R])
    return out + ((D, acc) if return_planes else ())


def tc_bound(X, V):
    """2 N 2^-57 max|b| max|x| + |exact| 2^-51 per column b of V [R, N] (the tc error bound, before the division)."""
    N = X.shape[0]
    mx = np.abs(X).max()
    return 2 * N * TC_BOUND * np.abs(V).max(axis=1) * mx


def scales(X):
    """scales_kernel: sqrt of fma-accumulated sum of squares (exact for integer designs below 2^53), 1 for a zero column."""
    z = (np.asarray(X, np.float64) ** 2).sum(axis=0)
    z[z == 0] = 1.0
    return np.sqrt(z)


def epis_pairs(K):
    """Candidate numbering of include/pareben.h: 0..K-1 main effects (i, i), then pairs i < j row-major."""
    I = list(range(K)); J = list(range(K))
    for i in range(K):
        for j in range(i + 1, K):
            I.append(i); J.append(j)
    return np.array(I), np.array(J)


def epis_columns(X):
    I, J = epis_pairs(X.shape[1])
    return np.where(I == J, X[:, I], X[:, I] * X[:, J])


# ---------------------------------------------------------------------------------------------------------------------
# right-hand-side columns of the kinds where digit extraction goes wrong

RHS_KINDS = ("normal", "zero", "single", "pow2_max", "neg_max", "span80", "tiny")


def rhs_column(rng, N, kind):
    if kind == "normal":
        return rng.normal(size=N)
    if kind == "zero":
        return np.zeros(N)
    if kind == "single":
        v = np.zeros(N); v[rng.integers(N)] = rng.normal() * 3.0
        return v
    if kind == "pow2_max":              # the maximum is exactly 2^5: frexp puts it at the top of its binade
        v = rng.uniform(-31.9, 31.9, N); v[rng.integers(N)] = 32.0
        return v
    if kind == "neg_max":
        v = rng.uniform(-1.0, 1.0, N); v[rng.integers(N)] = -1.75
        return v
    if kind == "span80":                # 2^-40 .. 2^40 within one column, both signs
        return rng.choice([-1.0, 1.0], N) * np.ldexp(rng.uniform(1.0, 2.0, N), rng.integers(-40, 40, N))
    if kind == "tiny":                  # max <= 1e-290: the documented exception, contributes exactly 0
        return rng.uniform(-1.0, 1.0, N) * 1e-291
    raise ValueError(kind)


def design(rng, N, K, codes):
    return rng.choice(np.asarray(codes, np.float64), size=(N, K))


# ---------------------------------------------------------------------------------------------------------------------
# tests of the references themselves

def _fraction_dot(a, b):
    return sum((Fraction(float(x)) * Fraction(float(y)) for x, y in zip(a, b)), Fraction(0))


@pytest.mark.parametrize("kind", ["int", "real", "wide"])
def test_exact_dot_matches_fractions(kind):
    rng = np.random.default_rng({"int": 1, "real": 2, "wide": 3}[kind])
    N, K, R = 37, 5, 4
    A = design(rng, N, K, [-127, -3, 0, 1, 127]) if kind == "int" else rng.normal(size=(N, K)) * 3.7
    B = np.stack([rhs_column(rng, N, k) for k in ("normal", "span80", "pow2_max", "single")], axis=1)
    if kind == "wide":
        B[:, 0] *= 2.0 ** 900
        B[3, 2] = 1.5 * 2.0 ** 950
    hi, lo = exact_dot(A, B)
    for r in range(R):
        for c in range(K):
            ex = _fraction_dot(A[:, c], B[:, r])
            assert hi[r, c] == float(ex)
            assert abs(Fraction(hi[r, c]) + Fraction(lo[r, c]) - ex) <= abs(ex) * Fraction(2) ** -104


def test_digits_are_balanced_and_exact():
    rng = np.random.default_rng(4)
    top = 2 ** 55 - 1
    q = np.concatenate([rng.integers(-top, top, 20000), [0, 1, -1, 63, 64, 65, -64, -65, top, -top, 2 ** 54 + 64, -(2 ** 54) - 64,
                                                         2 ** 28 - 1, 2 ** 28, -(2 ** 28), 2 ** 55 - 2 ** 28]])
    D = tc_digits(q)
    assert D.min() >= -64 and D.max() <= 64
    rec = np.zeros_like(q)
    for s in range(8):
        rec = rec * 128 + D[s]
    assert np.array_equal(rec, q)
    # w = (2^54 + 64) 2^-60 is q = 2^54 + 64 after scaling: its least significant plane is -64
    assert list(tc_digits(np.array([2 ** 54 + 64]))[:, 0]) == [32, 0, 0, 0, 0, 0, 1, -64]


def _check_tc_emulation(X, phi, w, e):
    N = X.shape[0]
    G, bb, ze = tc_emulate(X, phi, w, e)
    V = np.concatenate([w[None, :] * phi, e[None, :]], axis=0)
    hi, lo = exact_dot(X, V.T)
    err = err_vs(np.concatenate([G, ze[None, :]]), hi, lo)
    bound = tc_bound(X, V)[:, None] + np.abs(hi) * 2.0 ** -51
    assert np.all(err <= bound), f"max error/bound {np.max(err / np.maximum(bound, 1e-300)):.3g}"
    hb, lb = exact_dot(X * X, V[0][:, None])
    eb = err_vs(bb, hb[0], lb[0])
    assert np.all(eb <= 2 * N * TC_BOUND * np.abs(V[0]).max() * np.abs(X).max() ** 2 + np.abs(hb[0]) * 2.0 ** -51)
    return G, bb, ze


@pytest.mark.parametrize("N,K,codes", [(2, 3, [0, 1, 2]), (33, 7, [-1, 0, 1]), (400, 9, [-11, 0, 11]), (1089, 5, [-11, -1, 0, 1, 11])])
def test_tc_emulation_within_bound(N, K, codes):
    rng = np.random.default_rng(N)
    X = design(rng, N, K, codes)
    kinds = [k for k in RHS_KINDS if k != "tiny"]
    w = np.ldexp(1.0, -rng.integers(2, 7, N)) * rng.uniform(0.5, 1.0, N)
    phi = np.stack([np.ones(N)] + [rhs_column(rng, N, k) for k in kinds])
    e = rhs_column(rng, N, "span80")
    _check_tc_emulation(X, phi, w, e)


def test_tc_emulation_tiny_column_is_zero():
    rng = np.random.default_rng(5)
    N = 61
    X = design(rng, N, 4, [-11, 0, 11])
    w = np.full(N, 0.25)
    phi = np.stack([np.ones(N), rhs_column(rng, N, "tiny") * 4.0])
    G, bb, ze = tc_emulate(X, phi, w, rhs_column(rng, N, "tiny"))
    assert np.all(G[1] == 0) and np.all(ze == 0)
    assert np.all(G[0] != 0)


def test_tc_emulation_column_max_above_2_1022():
    """A column whose largest entry is >= 2^1022 scales by 2^(ex+1) = 2^1024 or 2^1025: split as 2^-5 / 2^-7 in Horner's
    last step and 2^(ex-1) the result is the exact dot product to the usual bound, where 2^(ex+1) as a double is +Inf."""
    rng = np.random.default_rng(6)
    N = 45
    X = design(rng, N, 6, [0, 1, 2])
    X[7, :] = [0, 1, 1, 0, 1, 0]
    w = np.ones(N)
    big = rng.uniform(-1.0, 1.0, N) * 2.0 ** 1000
    big[7] = 1.5 * 2.0 ** 1022
    phi = np.stack([np.ones(N), big])
    e = rng.uniform(-1, 1, N) * 2.0 ** 1010
    e[7] = -(2.0 ** 1023) * 1.25
    G, bb, ze = _check_tc_emulation(X, phi, w, e)
    assert np.all(np.isfinite(G)) and np.all(np.isfinite(ze))
    assert G[1, 1] != 0 and abs(G[1, 1]) > 2.0 ** 1021


def test_epis_numbering():
    I, J = epis_pairs(5)
    assert list(zip(I[5:], J[5:]))[:5] == [(0, 1), (0, 2), (0, 3), (0, 4), (1, 2)]
    K = 16
    I, J = epis_pairs(K)
    for c in range(K, I.size):
        i, j = I[c], J[c]
        assert c == K + i * (2 * K - i - 1) // 2 + (j - i - 1)
