"""GPU suite (-m gpu): the score contractions kernel by kernel, against exact references.

A module fixture compiles tests/kernels/contract_probe.cu (the library's own headers, __graft_entry__.NVCC_FLAGS) into
build/probe/ and loads it with ctypes.  The probe lays the design out with the library's layout kernels and runs one
block of tc_contract or contract_x with the fit kernels' resources.

* tc_contract (int8 tensor cores) must equal the numpy emulation of test_contract_reference.py bit for bit, and be
  within 2 N 2^-57 max|b| max|x| + |exact| 2^-51 of the exact value before the division by the column norm.
* contract_x (FP64: contract_col, contract_simt, DMMA) must be within (N + 4) 2^-53 sum|x||b| / s_c of the exact value,
  and give bitwise the same results for int8 and f64 operands of an integer design.
* Both: exact duplicate candidates tie bitwise, and a right-hand side's outputs do not depend on how many others share
  the contraction.
Every assertion message names the kernel, the shape and the largest error/bound ratio.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest

import test_contract_reference as ref

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PROBE_SRC = os.path.join(ROOT, "tests", "kernels", "contract_probe.cu")
CSRC = os.path.join(ROOT, "pareben_b200", "csrc")
U = 2.0 ** -53

_d = ctypes.POINTER(ctypes.c_double)
_i = ctypes.POINTER(ctypes.c_int)


@pytest.fixture(scope="module")
def probe():
    import shutil
    import __graft_entry__ as ge
    import pareben_b200 as pb
    if pb.device_count() < 1:
        pytest.fail("no CUDA device: the -m gpu suite must run on the B200 box")
    out_dir = os.path.join(ROOT, "build", "probe")
    lib = os.path.join(out_dir, "libcontract_probe.so")
    sources = [PROBE_SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(ROOT, "__graft_entry__.py")]
    if not ge._newer(lib, sources):
        os.makedirs(out_dir, exist_ok=True)
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        subprocess.run([nvcc, *ge.NVCC_FLAGS, "--shared", "-o", lib, PROBE_SRC], check=True, cwd=out_dir)
    L = ctypes.CDLL(lib)
    L.probe_tc.argtypes = [ctypes.c_int, ctypes.c_int, _d, ctypes.c_int, _d, _d, _d, _d, _d, _d, _d]
    L.probe_contract_x.argtypes = [ctypes.c_int] * 5 + [_d, ctypes.c_int, _d, _d, _d, ctypes.c_int, _d, _d, _d, _d]
    L.probe_cand_map.argtypes = [ctypes.c_int, ctypes.c_int, _i, _i]
    L.probe_last_error.restype = ctypes.c_char_p
    return L


def _p(a):
    return None if a is None else a.ctypes.data_as(_d)


def _c(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def run_tc(L, X, phi, w, e):
    """tc_contract on X [N, K], phi [R, N], w, e [N] -> (G [R, K], bb, ze, scale)."""
    X = _c(X); N, K = X.shape
    phi = _c(np.asarray(phi).reshape(-1, N)); R = phi.shape[0]
    G = np.full((max(R, 1), K), np.nan); bb = np.full(K, np.nan); ze = np.full(K, np.nan); sc = np.full(K, np.nan)
    rc = L.probe_tc(N, K, _p(X), R, _p(phi), _p(_c(w)), _p(_c(e)), _p(G), _p(bb), _p(ze), _p(sc))
    assert rc == 0, f"probe_tc: {rc} {L.probe_last_error().decode()}"
    return G[:R], bb, ze, sc


def run_cx(L, X, cols, epis=False, force_f64=False, n_aligned=None, w=None, e=None, want_bb=False):
    """contract_x on X [N, K], cols [R, N] -> (G [R, Kc], bb, ze, scale)."""
    X = _c(X); N, K = X.shape
    cols = _c(cols); R = cols.shape[0]
    Kc = K * (K + 1) // 2 if epis else K
    n_aligned = R if n_aligned is None else n_aligned
    G = np.full((R, Kc), np.nan); bb = np.full(Kc, np.nan); ze = np.full(Kc, np.nan); sc = np.full(Kc, np.nan)
    rc = L.probe_contract_x(N, K, int(epis), int(force_f64), n_aligned, _p(X), R, _p(cols),
                            _p(None if w is None else _c(w)), _p(None if e is None else _c(e)), int(want_bb),
                            _p(G), _p(bb), _p(ze), _p(sc))
    assert rc == 0, f"probe_contract_x: {rc} {L.probe_last_error().decode()}"
    return G, bb, ze, sc


def bits_equal(a, b):
    """Bitwise equal (so +0 and -0 differ); any NaN equals any NaN (payloads are not part of the result)."""
    a = np.ascontiguousarray(a, np.float64); b = np.ascontiguousarray(b, np.float64)
    if a.shape != b.shape:
        return False
    nan = np.isnan(a)
    return np.array_equal(nan, np.isnan(b)) and np.array_equal(a[~nan].view(np.int64), b[~nan].view(np.int64))


# ---------------------------------------------------------------------------------------------------------------------
# tc_contract

CODES = {"012": [0, 1, 2], "pm1": [-1, 0, 1], "11": [-11, 0, 11]}


def tc_inputs(rng, N, K, R1, codes):
    """A design with an all-zero candidate and exact duplicates in different 128-candidate tiles, and R1 right-hand-side
    columns (w o phi_j, then e) cycling through the kinds of ref.RHS_KINDS.  w is a power of two per row (<= 1/4, as
    IRLS weights are), so that b = w o phi has exactly the kind asked for."""
    X = ref.design(rng, N, K, CODES[codes])
    if K > 2:
        X[:, 1] = 0.0
    for a, b in ((0, 130), (2, 300), (129, 257), (3, 128)):
        if b < K:
            X[:, b] = X[:, a]
    w = np.ldexp(1.0, -rng.integers(2, 7, N))
    B = [ref.rhs_column(rng, N, ref.RHS_KINDS[j % len(ref.RHS_KINDS)]) for j in range(R1)]
    phi = np.stack([np.ones(N)] + [B[j] / w for j in range(1, R1 - 1)]) if R1 > 1 else np.zeros((0, N))
    e = B[-1] if R1 > 1 else B[0]
    return X, phi, w, e


def check_tc(L, X, phi, w, e, what):
    N, K = X.shape
    G, bb, ze, sc = run_tc(L, X, phi, w, e)
    eG, ebb, eze = ref.tc_emulate(X, phi, w, e, scale=sc)
    assert bits_equal(sc, ref.scales(X)), f"{what}: column norms differ from sqrt(sum x^2)"
    for name, got, want in (("G", G, eG), ("bb", bb, ebb), ("ze", ze, eze)):
        if not bits_equal(got, want):
            bad = np.argwhere(~(((got == want) & (np.signbit(got) == np.signbit(want))) | (np.isnan(got) & np.isnan(want))))
            raise AssertionError(f"tc_contract {what}: {name} differs from the emulation at {len(bad)} entries, first {bad[:3].tolist()}: "
                                 f"{got[tuple(bad[0])]!r} vs {want[tuple(bad[0])]!r}")
    # within the bound of the exact value (finite columns only)
    V = np.concatenate([w[None, :] * phi, e[None, :]])
    fin = np.all(np.isfinite(V), axis=1)
    tiny = fin & (np.abs(V).max(axis=1) <= 1e-290)      # the documented exception: such a column contributes exactly 0
    assert np.all(np.concatenate([G, ze[None, :]])[tiny] == 0), f"tc_contract {what}: a column with max <= 1e-290 is not 0"
    fin &= ~tiny
    hi, lo = ref.exact_dot(X, np.where(fin[:, None], V, 0.0).T)
    pre, _, _ = ref.tc_emulate(X, phi, w, e)
    err = ref.err_vs(np.concatenate([pre, ze[None, :]]), hi, lo)
    bound = ref.tc_bound(X, np.where(fin[:, None], V, 0.0))[:, None] + np.abs(hi) * 2.0 ** -51
    ratio = np.where(fin[:, None], err / np.maximum(bound, 1e-300), 0.0)
    assert ratio.max() <= 1.0, f"tc_contract {what}: error/bound {ratio.max():.3g}"
    if phi.shape[0] > 0:        # after the division by s_c: the bound / s_c plus one rounding
        R = phi.shape[0]
        errd = ref.err_vs(G[fin[:R]], hi[:R][fin[:R]], lo[:R][fin[:R]], scale=sc)
        bd = bound[:R][fin[:R]] / sc[None, :] + np.abs(G[fin[:R]]) * 2.0 ** -52
        r2 = (errd / np.maximum(bd, 1e-300)).max() if errd.size else 0.0
        assert r2 <= 1.0, f"tc_contract {what}: error/bound after the division {r2:.3g}"
    return G, bb, ze, ratio.max()


TC_CASES = [  # N, Kc, R + 1, codes
    (2, 1, 1, "012"), (3, 127, 2, "pm1"), (31, 128, 29, "11"), (32, 129, 30, "012"), (33, 256, 31, "pm1"),
    (61, 300, 59, "11"), (400, 481, 60, "012"), (1089, 300, 61, "pm1"), (400, 129, 91, "11"), (1089, 481, 31, "11"),
    (33, 1, 91, "012"), (61, 128, 2, "11"),
]


@pytest.mark.parametrize("N,K,R1,codes", TC_CASES)
def test_tc_contract_matches_emulation(probe, N, K, R1, codes):
    rng = np.random.default_rng(N * 1000 + K + R1)
    X, phi, w, e = tc_inputs(rng, N, K, R1, codes)
    G, bb, ze, worst = check_tc(probe, X, phi, w, e, f"N={N} Kc={K} R+1={R1} codes={codes}")
    for a, b in ((0, 130), (2, 300), (129, 257), (3, 128)):
        if b < K:
            assert bits_equal(G[:, a], G[:, b]) and bits_equal(bb[a], bb[b]) and bits_equal(ze[a], ze[b]), \
                f"tc_contract N={N} Kc={K}: duplicate candidates {a} and {b} do not tie"


def test_tc_contract_rows_do_not_depend_on_R_or_candidate_order(probe):
    """A right-hand side's G row is the same whichever pass of 30 columns it falls in, and a candidate's outputs are the
    same wherever the candidate sits among the 128-candidate tiles."""
    rng = np.random.default_rng(11)
    N, K = 333, 300
    X, phi, w, e = tc_inputs(rng, N, K, 91, "pm1")
    G, bb, ze, _ = run_tc(probe, X, phi, w, e)
    for R in (1, 2, 29, 30, 31, 59, 61):
        g, b2, _, _ = run_tc(probe, X, phi[:R], w, e)
        assert bits_equal(g, G[:R]) and bits_equal(b2, bb), f"tc_contract N={N}: G rows change with R = {R}"
    perm = rng.permutation(K)
    g, b2, z2, _ = run_tc(probe, X[:, perm], phi, w, e)
    assert bits_equal(g, G[:, perm]) and bits_equal(b2, bb[perm]) and bits_equal(z2, ze[perm]), \
        "tc_contract: outputs change when the candidates are permuted across tiles"


def test_tc_contract_nonfinite_column_is_contained(probe):
    """A NaN or Inf in one phi column makes that column's outputs NaN and leaves every other column bitwise unchanged."""
    rng = np.random.default_rng(12)
    N, K = 97, 200
    X, phi, w, e = tc_inputs(rng, N, K, 35, "11")
    G, bb, ze, _ = run_tc(probe, X, phi, w, e)
    bad = phi.copy()
    bad[3, 50] = np.nan
    bad[31, 7] = np.inf
    g, b2, z2, _ = check_tc(probe, X, bad, w, e, "NaN / Inf columns")
    assert np.all(np.isnan(g[3])) and np.all(np.isnan(g[31]))
    keep = [j for j in range(phi.shape[0]) if j not in (3, 31)]
    assert bits_equal(g[keep], G[keep]) and bits_equal(b2, bb) and bits_equal(z2, ze)


def test_tc_contract_column_max_above_2_1022(probe):
    """Right-hand sides whose largest entry is >= 2^1022 (in a phi column and in e): finite, exact to the bound."""
    rng = np.random.default_rng(13)
    N, K = 70, 140
    X = ref.design(rng, N, K, [0, 1, 2])
    X[9] = rng.choice([0.0, 1.0], K)
    w = np.ones(N)
    big = rng.uniform(-1.0, 1.0, N) * 2.0 ** 1000
    big[9] = 1.5 * 2.0 ** 1022
    phi = np.stack([np.ones(N), big, rng.normal(size=N)])
    e = rng.uniform(-1.0, 1.0, N) * 2.0 ** 1010
    e[9] = -1.25 * 2.0 ** 1023
    G, bb, ze, _ = check_tc(probe, X, phi, w, e, "column max >= 2^1022")
    assert np.all(np.isfinite(G)) and np.all(np.isfinite(ze))


def test_tc_contract_int32_headroom(probe):
    """The largest training-row count the host predicate n max|x|^2 64 < 2^31 admits at |x| = 11: with w = (2^54 + 64)
    2^-60 every row's least significant digit is -64, so bb's plane sum is -64 121 N = -2,147,480,896, just inside int32."""
    N = 277_309
    assert N * 121 * 64 < 2 ** 31 <= (N + 1) * 121 * 64
    rng = np.random.default_rng(14)
    X = rng.choice([-11.0, 11.0], size=(N, 1))
    w = np.full(N, (2.0 ** 54 + 64) * 2.0 ** -60)
    e = rng.uniform(-1.0, 1.0, N)
    phi = np.ones((1, N))
    _, _, _, D, _ = ref.tc_emulate(X, phi, w, e, return_planes=True)
    assert np.all(D[7, 0] == -64) and int((D[7, 0] * 121).sum()) == -2_147_480_896
    G, bb, ze, _ = check_tc(probe, X, phi, w, e, f"N={N} |x|=11")
    assert bb[0] == float(121 * N * (2 ** 54 + 64)) * 2.0 ** -60


def test_tc_host_predicate_row_limit(built):
    """At library level a binomial ±11 design takes the tensor-core path up to n = 277,309 rows, and not at 277,310."""
    import pareben_b200 as pb
    if pb.device_count() < 1:
        pytest.fail("no CUDA device")
    rng = np.random.default_rng(15)
    for n, tc in ((277_309, True), (277_310, False)):
        X = rng.choice([-11.0, 0.0, 11.0], size=(n, 2))
        y = (rng.random(n) < 0.5).astype(np.float64)
        with pb.Problem(X, y, None, 0, False, "binomial") as p:
            assert p.contraction_info()[0] is tc, f"n = {n}: tensor-core path {p.contraction_info()[0]}, expected {tc}"


# ---------------------------------------------------------------------------------------------------------------------
# contract_x

def cx_design(rng, N, K, kind):
    if kind == "pm1":
        return ref.design(rng, N, K, [-1, 0, 1])
    if kind == "i127":
        X = rng.integers(-127, 128, size=(N, K)).astype(np.float64)
        X[0, 0] = 127.0; X[min(1, N - 1), min(1, K - 1)] = -127.0
        return X
    return rng.normal(size=(N, K)) * rng.uniform(0.5, 2.0, K)


def cx_form(N, R, want_bb):
    ldt = (N + 63) & ~63
    if R == 1 and not want_bb and ldt <= 5120:
        return "contract_col"
    if R <= 4 and not want_bb:
        return "contract_simt"
    return "contract_mma"


CX_CASES = [  # N, K, epis, design, R, n_aligned, weights ("", "w" or "wbb")
    (2, 1, False, "pm1", 1, 1, ""),
    (17, 127, False, "i127", 2, 2, "w"),
    (64, 128, False, "real", 4, 4, ""),
    (65, 129, False, "pm1", 5, 5, "wbb"),
    (1087, 256, False, "i127", 9, 9, ""),
    (1088, 257, False, "pm1", 1, 0, "w"),
    (1089, 128, False, "i127", 3, 3, ""),
    (5120, 129, False, "i127", 1, 1, ""),
    (5121, 129, False, "i127", 1, 1, ""),
    (6000, 64, False, "real", 1, 0, "w"),
    (6000, 40, False, "pm1", 33, 33, "wbb"),
    (400, 300, False, "i127", 31, 20, ""),
    (300, 200, False, "real", 32, 32, "wbb"),
    (200, 100, False, "pm1", 64, 0, ""),
    (150, 129, False, "i127", 65, 60, "wbb"),
    (333, 128, False, "pm1", 8, 3, "wbb"),
    (200, 15, True, "i127", 1, 1, ""),
    (1089, 16, True, "pm1", 4, 4, "w"),
    (100, 16, True, "i127", 9, 9, "wbb"),
    (77, 15, True, "real", 33, 30, ""),
    (5121, 16, True, "pm1", 1, 1, ""),
]


def cx_inputs(rng, N, K, design, R, weights):
    X = cx_design(rng, N, K, design)
    if K >= 3:
        X[:, K - 1] = X[:, 0]                  # an exact duplicate candidate (and, for Epis, duplicate pairs)
    cols = np.stack([ref.rhs_column(rng, N, ("normal", "span80", "pow2_max", "neg_max", "single")[r % 5]) for r in range(R)])
    w = rng.uniform(0.01, 0.25, N) if weights else None
    e = rng.normal(size=N) if weights == "wbb" else None
    return X, cols, w, e


def check_cx(L, X, cols, epis, n_aligned, w, e, want_bb, what):
    N, K = X.shape
    A = ref.epis_columns(X) if epis else X
    G, bb, ze, sc = run_cx(L, X, cols, epis, False, n_aligned, w, e, want_bb)
    assert bits_equal(sc, ref.scales(A)) or np.allclose(sc, ref.scales(A), rtol=1e-15), f"{what}: column norms"
    B = cols if w is None else cols * w[None, :]
    hi, lo = ref.exact_dot(A, B.T)
    err = ref.err_vs(G, hi, lo, scale=sc)
    bound = (N + 4) * U * ref.abs_dot(A, B.T) / sc[None, :]
    ratios = [(err / np.maximum(bound, 1e-300)).max()]
    assert ratios[0] <= 1.0, f"{what}: G error/bound {ratios[0]:.3g}"
    if want_bb:
        for name, got, AA, b in (("bb", bb, A * A, w), ("ze", ze, A, e)):
            h, l = ref.exact_dot(AA, b[:, None])
            r = (ref.err_vs(got, h[0], l[0]) / np.maximum((N + 4) * U * ref.abs_dot(AA, b[:, None])[0], 1e-300)).max()
            assert r <= 1.0, f"{what}: {name} error/bound {r:.3g}"
            ratios.append(r)
    return G, bb, ze, max(ratios)


@pytest.mark.parametrize("N,K,epis,design,R,n_aligned,weights", CX_CASES)
def test_contract_x_within_bound(probe, N, K, epis, design, R, n_aligned, weights):
    rng = np.random.default_rng(N * 7 + K * 3 + R)
    X, cols, w, e = cx_inputs(rng, N, K, design, R, weights)
    want_bb = weights == "wbb"
    form = cx_form(N, R, want_bb)
    what = f"{form} ({'Epis' if epis else 'main'}) N={N} K={K} R={R} n_aligned={n_aligned} design={design} weights={weights or '-'}"
    G, bb, ze, worst = check_cx(probe, X, cols, epis, n_aligned, w, e, want_bb, what)
    print(f"{what}: max error/bound {worst:.3g}")
    Kc = G.shape[1]
    if K >= 3:      # the duplicate candidate K-1 of 0, and for Epis the pairs (i, K-1) of (0, i)
        dup = [(0, K - 1)]
        if epis:
            I, J = ref.epis_pairs(K)
            idx = {(i, j): c for c, (i, j) in enumerate(zip(I, J))}
            dup += [(idx[(0, i)], idx[(i, K - 1)]) for i in range(1, K - 1)]
        for a, b in dup:
            assert bits_equal(G[:, a], G[:, b]), f"{what}: duplicate candidates {a} and {b} do not tie"
            if want_bb:
                assert bits_equal(bb[a], bb[b]) and bits_equal(ze[a], ze[b]), f"{what}: duplicate bb / ze do not tie"
    if design != "real":        # int8 and f64 operands: widening is exact and the FMA order is the same
        G2, bb2, ze2, _ = run_cx(probe, X, cols, epis, True, n_aligned, w, e, want_bb)
        assert bits_equal(G2, G), f"{what}: int8 and f64 operands differ"
        if want_bb:
            assert bits_equal(bb2, bb) and bits_equal(ze2, ze), f"{what}: int8 and f64 operands differ in bb / ze"
    # fewer right-hand sides in the same form: the rows that remain are unchanged
    for R2 in (r for r in (1, 2, 4, 5, 8, 9, 31, 32, 33) if r < R and cx_form(N, r, want_bb) == form):
        G3, bb3, ze3, _ = run_cx(probe, X, cols[:R2], epis, False, min(n_aligned, R2), w, e, want_bb)
        assert bits_equal(G3, G[:R2]), f"{what}: rows change when R drops to {R2}"
        if want_bb:
            assert bits_equal(bb3, bb) and bits_equal(ze3, ze), f"{what}: bb / ze change when R drops to {R2}"
    assert Kc == (K * (K + 1) // 2 if epis else K)


def test_epis_candidate_numbering(probe):
    """The kernels' candidate decoding (Cand<true>) is the numbering documented in include/pareben.h."""
    for K in (1, 2, 15, 16, 300):
        Kc = K * (K + 1) // 2
        I = np.zeros(Kc, np.int32); J = np.zeros(Kc, np.int32)
        assert probe.probe_cand_map(K, Kc, I.ctypes.data_as(_i), J.ctypes.data_as(_i)) == 0
        eI, eJ = ref.epis_pairs(K)
        assert np.array_equal(I, eI) and np.array_equal(J, eJ), f"K={K}: candidate numbering differs"
