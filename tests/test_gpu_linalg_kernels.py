"""GPU suite (-m gpu): the dense linear algebra of a fit kernel by kernel, against the references of
test_linalg_reference.py.

A module fixture compiles tests/kernels/linalg_probe.cu (the library's own headers, __graft_entry__.NVCC_FLAGS with
-fmad=false) into build/probe/ and loads it with ctypes (kernel_probe.py).  Every probe call runs one block with the fit
kernels' resources, every device buffer sits between guard regions (a write past either end fails the call), and the
emit / out callbacks count their calls: every candidate and every pair j <= k must come out exactly once.

Sizes come from the dispatch constants the probe exports, so the boundaries move with them:
  spd_inverse_sweep   sweep_regs<1> (M <= 32), sweep_regs<2> (M <= SWEEP_SMEM_M), sweep_panel with 8-wide panels while
                      16 Mp + 8 <= SWEEP_PANEL_DOUBLES and 4-wide while 8 Mp + 8 fits (Mp = M rounded up to 8, + 4),
                      sweep_core above;
  quad_forms          quad_forms_simt<8> up to QUAD_SIMT_M, then quad_forms_mma: every width of the last 32-column chunk,
                      and M = 784 / 785 where the cache row offsets stop fitting in shared memory;
  gram                gram_pipe up to PHIT_LD columns, gram_mma above.

Checks:
1. Bit for bit against the C restatements: sweep_regs<1/2>, sweep_core, quad_forms_simt (quad and lin, with an
   asymmetric SIGMA so that the triangle read is pinned), gram_pipe (H and the gradient), cache_dot, sym_matvec_row.
2. Exactly the exact answer on the certified exact cases, on every path: both panel widths, quad_forms_mma, gram_mma.
3. Within a bound on realistic inputs (H = PHI'B PHI + diag(0, alpha), test_linalg_reference.hessian):
   * g'SIGMA g.  quad = sum_p g_p z_p with z_p = sum_{j<=p} g_j sigma'_jp.  A term g_j sigma'_jp g_p passes through at
     most p - j + 4 roundings in z_p (a DMMA k-step adds four products, in an unspecified order) and at most
     M/4 + 3 in the sum over p (a lane's chain, then two shuffles), so |error| <= gamma_(M+8) sum |terms|
     = (M + 8) u |g|'|SIGMA||g| to first order (sum over j <= p of |sigma'| is |SIGMA| for a symmetric SIGMA).  lin the
     same with |g|'|v|.
   * H = PHI'B PHI.  gram_mma forms fl(phi_j w) first, then one DMMA accumulator chain over the N rows (one row split
     for M > 64): each term passes through at most N roundings, so |error| <= (N + 4) u sum_h |fl(phi_j w)| |phi_k|.
   * A^-1.  The sweep is Gauss-Jordan elimination with diagonal pivots; for a symmetric positive definite A it is
     forward stable (Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., section 14.4):
     ||X - A^-1|| <= c_M u kappa(A) ||A^-1|| with c_M of modest degree in M.  The test takes
     ||X - A^-1||_2 <= 2 M u kappa_2(A) ||A^-1||_2.
   The references carry errors at least 2^8 below these bounds (test_linalg_reference.py).
4. Invariants, bitwise, on every path: the inverse is exactly symmetric; power-of-two diagonal scaling commutes,
   inv(DAD) = D^-1 inv(A) D^-1 with D over 2^+-30; duplicate candidates tie in the quadratic forms (positions that
   differ mod 8, different 128-candidate rounds, both lanes of the SIMT pair, both tiles of a warp); outputs follow a
   candidate permutation and do not depend on the physical row order grow.
5. Failure: a pivot exactly zero, negative or NaN at k = 0, at a panel's first column, mid-panel and at k = M - 1 makes
   ok false in all FIT_T threads, with the guards intact (what a failed sweep leaves in a is not pinned).
Every assertion message names the path, the shape and the worst error/bound ratio where there is one.
"""
import ctypes
import functools
from types import SimpleNamespace

import numpy as np
import pytest

import kernel_probe as kp
import test_linalg_reference as ref
from kernel_probe import bits_equal, dp, f64, ip

pytestmark = pytest.mark.gpu

CONSTANTS = ("SWEEP_SMEM_M", "SWEEP_PANEL_DOUBLES", "QUAD_SIMT_M", "QT", "PHIT_LD", "FIT_T")
ROWOFF_M = 784          # quad_forms_mma keeps the cache row offsets in shared memory up to this M
BASIS_CAP = 1024        # the library's default basis cap


@pytest.fixture(scope="module")
def P():
    L = kp.build_probe("linalg_probe")
    d, i = kp.D, ctypes.c_int
    L.probe_last_error.restype = ctypes.c_char_p
    L.probe_constant.restype = ctypes.c_longlong
    L.probe_constant.argtypes = [ctypes.c_char_p]
    L.probe_sweep.argtypes = [i, d, kp.I]
    L.probe_quad.argtypes = [i, i, i, kp.I, d, d, d, d, d, kp.I]
    L.probe_gram.argtypes = [i, i, i, d, d, d, d, kp.I, d, kp.I]
    L.probe_cache_dot.argtypes = [i, i, i, kp.I, d, d, d, kp.I]
    L.probe_sym_matvec.argtypes = [i, d, d, d]
    if L.probe_device_count() < 1:
        pytest.fail("no CUDA device: the -m gpu suite must run on the B200 box")
    C = {n: int(L.probe_constant(n.encode())) for n in CONSTANTS}
    assert min(C.values()) > 0, C
    return SimpleNamespace(L=L, C=C)


def _check(P, rc, what):
    assert rc == 0, f"{what}: probe returned {rc}: {P.L.probe_last_error().decode()}"


# ---------------------------------------------------------------------------------------------------------------------
# probe wrappers

def run_sweep(P, A):
    """(ok flags [FIT_T], a as the kernel leaves it) for the symmetric M x M matrix A."""
    a = f64(np.array(A, dtype=np.float64, copy=True))
    ok = np.full(P.C["FIT_T"], -7, np.int32)
    _check(P, P.L.probe_sweep(a.shape[0], dp(a), ip(ok)), f"sweep M={a.shape[0]}")
    return ok, a


def physical(rng, G, extra=5):
    """(grow, Gphys): the logical rows of G scattered over M + extra physical rows; the unused rows are NaN."""
    M, Kc = G.shape
    grow = rng.permutation(M + extra)[:M].astype(np.int32)
    Gp = np.full((M + extra, Kc), np.nan)
    Gp[grow] = G
    return grow, Gp


def run_quad(P, G, sigma, v=None, rng=None, grow=None):
    """(quad, lin) for logical cache rows G [M, Kc]; asserts one emit per candidate."""
    M, Kc = G.shape
    if grow is None:
        grow, Gp = physical(rng if rng is not None else np.random.default_rng(M), G)
    else:
        Gp = np.full((int(grow.max()) + 1, Kc), np.nan); Gp[grow] = G
    q = np.full(Kc, np.nan); l = np.full(Kc, np.nan); cnt = np.zeros(Kc, np.int32)
    _check(P, P.L.probe_quad(M, Kc, Gp.shape[0], ip(grow), dp(f64(Gp)), dp(f64(sigma)), dp(None if v is None else f64(v)),
                             dp(q), dp(l), ip(cnt)), f"quad_forms M={M} Kc={Kc}")
    assert np.all(cnt == 1), f"quad_forms M={M} Kc={Kc}: emit counts {np.unique(cnt)}"
    return q, l


def run_gram(P, phi, w=None, ev=None, mma=False):
    """H [M, M] (j <= k filled, NaN below) and g [M] (gram_pipe with ev); asserts one call per pair and per column."""
    phi = f64(phi); M, N = phi.shape
    H = np.full((M, M), np.nan); cH = np.zeros((M, M), np.int32)
    g = np.full(M, np.nan) if ev is not None else None
    cg = np.zeros(M, np.int32) if ev is not None else None
    path = "gram_mma" if mma else "gram_pipe"
    _check(P, P.L.probe_gram(int(mma), N, M, dp(phi), dp(None if w is None else f64(w)), dp(None if ev is None else f64(ev)),
                             dp(H), ip(cH), dp(g), ip(cg)), f"{path} N={N} M={M}")
    assert np.array_equal(cH, np.triu(np.ones((M, M), np.int32))), f"{path} N={N} M={M}: out() not once per j <= k"
    if ev is not None:
        assert np.all(cg == 1), f"{path} N={N} M={M}: outg() not once per column"
    return H, g


def run_cache_dot(P, G, vec, rng):
    M, Kc = G.shape
    grow, Gp = physical(rng, G)
    z = np.full(Kc, np.nan); cnt = np.zeros(Kc, np.int32)
    _check(P, P.L.probe_cache_dot(M, Kc, Gp.shape[0], ip(grow), dp(f64(Gp)), dp(f64(vec)), dp(z), ip(cnt)), f"cache_dot M={M} Kc={Kc}")
    assert np.all(cnt == 1), f"cache_dot M={M} Kc={Kc}: emit counts {np.unique(cnt)}"
    return z


def run_sym_matvec(P, A, v):
    z = np.full(A.shape[0], np.nan)
    _check(P, P.L.probe_sym_matvec(A.shape[0], dp(f64(A)), dp(f64(v)), dp(z)), f"sym_matvec M={A.shape[0]}")
    return z


# ---------------------------------------------------------------------------------------------------------------------
# sizes from the constants

def sweep_paths(C):
    smem, pd = C["SWEEP_SMEM_M"], C["SWEEP_PANEL_DOUBLES"]
    mp = lambda M: ((M + 7) & ~7) + 4
    nb8 = max(M for M in range(smem + 1, 8192) if 16 * mp(M) + 8 <= pd)
    nb4 = max(M for M in range(smem + 1, 8192) if 8 * mp(M) + 8 <= pd)
    return {
        "regs1": [1, 2, 3, 31, 32],
        "regs2": [33, smem - 1, smem],
        "panel8": [smem + 1, smem + 8, smem + 9, nb8],
        "panel4": [nb8 + 1, nb4],
        "core": [nb4 + 1, max(BASIS_CAP, nb4 + 2)],
    }


SWEEP_PATHS = ("regs1", "regs2", "panel8", "panel4", "core")


@functools.lru_cache(maxsize=None)
def exact_inverse(M, seed=0):
    A, Ainv, D = ref.spd_exact(M, seed)
    if M not in ref.SWEEP_SIZES or seed:
        ok, piv, _ = ref.sweep_certificate(A)
        assert ok and np.array_equal(piv, D), f"M={M}: exact inverse case not certified"
    return A, Ainv


def quad_sizes(C):
    s = C["QUAD_SIMT_M"]
    simt = sorted({1, 2, 3, 7, 8, 9, 31, 32, 33, s - 1, s})
    mma = []
    for width in range(1, 5):                          # the last 32-column chunk holds `width` 8-column tiles
        Ms = [M for M in range(s + 1, s + 33) if ((M + 7) // 8 - 1) % 4 + 1 == width]
        mma += [Ms[0], Ms[-1]] if Ms else []
    mma = sorted(set(mma + [mma[-1] + 1, ROWOFF_M, ROWOFF_M + 1]))
    return simt, mma


KC_SIZES = (1, 7, 8, 9, 127, 128, 129, 511, 512, 513, 1100)


# ---------------------------------------------------------------------------------------------------------------------
# spd_inverse_sweep

@pytest.mark.parametrize("path", SWEEP_PATHS)
def test_sweep_exact(P, path):
    """Exact cases: the inverse must be exactly A^-1 on every path, exactly symmetric, ok in every thread."""
    for M in sweep_paths(P.C)[path]:
        A, Ainv = exact_inverse(M)
        ok, X = run_sweep(P, A)
        assert np.all(ok == 1), f"sweep {path} M={M}: ok flags {np.unique(ok)}"
        bad = np.count_nonzero(X != Ainv)
        assert bad == 0, f"sweep {path} M={M}: {bad} entries differ from the exact inverse (max |diff| {np.max(np.abs(X - Ainv)):.3g})"


@pytest.mark.parametrize("path", SWEEP_PATHS)
def test_sweep_realistic(P, path):
    """Realistic IRLS Hessians: bitwise against the C restatement (regs, core), within the normwise bound (all paths;
    the long-double reference is skipped above 700), exactly symmetric, and inv(DAD) = D^-1 inv(A) D^-1 bitwise."""
    worst = []
    for M in sweep_paths(P.C)[path]:
        rng = np.random.default_rng(1000 + M)
        _, _, A = ref.hessian(rng, max(64, 2 * M), M)
        ok, X = run_sweep(P, A)
        assert np.all(ok == 1), f"sweep {path} M={M}: ok flags {np.unique(ok)}"
        assert bits_equal(X, X.T), f"sweep {path} M={M}: inverse not exactly symmetric"
        if path != "panel8" and path != "panel4":
            cok, Xc = ref.c_sweep(A, core=(path == "core"))
            assert cok and bits_equal(X, Xc), \
                f"sweep {path} M={M}: {np.count_nonzero(X != Xc)} entries differ from the C restatement"
        if M <= 700:
            bound, _ = ref.inverse_bound(A)
            r = ref.inverse_err(X, A, ref.inverse_ref(A)) / bound
            worst.append((r, M))
            assert r <= 1.0, f"sweep {path} M={M}: ||X - A^-1||_2 / bound = {r:.3g}"
        e = rng.integers(-30, 31, M)
        d = np.ldexp(1.0, e)
        A2 = (A * d[:, None]) * d[None, :]
        ok2, X2 = run_sweep(P, A2)
        assert np.all(ok2 == 1)
        want = np.ldexp(np.ldexp(X, -e[:, None]), -e[None, :])
        assert bits_equal(X2, want), \
            f"sweep {path} M={M}: inv(DAD) != D^-1 inv(A) D^-1 in {np.count_nonzero(X2 != want)} entries"
    print(f"sweep {path}: worst error/bound {max(worst)[0]:.3g} at M={max(worst)[1]}" if worst else "")


@pytest.mark.parametrize("path", SWEEP_PATHS)
def test_sweep_failure(P, path):
    """A pivot exactly zero, negative or NaN at k = 0, a panel's first column, mid-panel and k = M - 1: ok is false in
    every thread and no guard is touched."""
    sizes = sweep_paths(P.C)[path]
    M = max(sizes) if path.startswith("regs") else (sizes[0] + sizes[-1]) // 2
    ks = sorted({0, 16 % M, 18 % M, M - 1}) if M > 1 else [0]
    for k in ks:
        for kind in ("zero", "neg", "nan"):
            A, _, _ = ref.spd_exact(M, 4, (k, kind))
            ok, _ = run_sweep(P, A)
            assert np.all(ok == 0), f"sweep {path} M={M}: {kind} pivot at k={k}: ok flags {np.unique(ok)}"


# ---------------------------------------------------------------------------------------------------------------------
# quad_forms

def _dups(Kc, T):
    """Candidate positions that carry copies of candidate 3: another position mod 8, the other tile of the warp, another
    128-candidate round, the SIMT pair partner and the next SIMT pass."""
    return [c for c in (3, 12, 67, 130, 3 + T, 3 + 2 * T, 1000) if c < Kc]


@pytest.mark.parametrize("kind", ["simt", "mma"])
def test_quad_exact(P, kind):
    """Small-integer G, dyadic SIGMA and v: quad and lin are exactly the exact values, for every Kc."""
    Ms = quad_sizes(P.C)[0 if kind == "simt" else 1]
    for M in Ms:
        for Kc in KC_SIZES:
            rng = np.random.default_rng([M, Kc])
            G = ref.int_cache(rng, M, Kc); S = ref.dyadic_sym(rng, M); v = ref.dyadic(rng, M)
            assert ref.quad_certificate(G, S, v)
            eq, el = ref.exact_quad_float(G, S, v)
            q, l = run_quad(P, G, S, v, rng)
            bq, bl = np.count_nonzero(q != eq), np.count_nonzero(l != el)
            assert bq == 0 and bl == 0, f"quad_forms_{kind} M={M} Kc={Kc}: {bq} quad and {bl} lin differ from the exact values"


def test_quad_simt_bitwise(P):
    """quad_forms_simt<8> against the C restatement, with an asymmetric SIGMA (the kernel reads sigma[p*M + j], j <= p)."""
    for M in quad_sizes(P.C)[0]:
        for Kc in KC_SIZES:
            rng = np.random.default_rng([M, Kc, 1])
            G = rng.normal(size=(M, Kc)); S = rng.normal(size=(M, M)); v = rng.normal(size=M)
            q, l = run_quad(P, G, S, v, rng)
            cq, cl = ref.c_quad(G, S, v)
            assert bits_equal(q, cq) and bits_equal(l, cl), \
                f"quad_forms_simt M={M} Kc={Kc}: {np.count_nonzero(q != cq)} quad, {np.count_nonzero(l != cl)} lin differ from C"
            q0, l0 = run_quad(P, G, S, None, rng)
            assert bits_equal(q0, cq) and np.all(l0 == 0), f"quad_forms_simt M={M} Kc={Kc}: v = null changes quad"


def test_quad_mma_within_bound(P):
    """quad_forms_mma on realistic inputs: SIGMA the inverse of an IRLS Hessian, G normal; (M + 8) u |g|'|SIGMA||g|."""
    worst = (0.0, (0, 0))
    for M in quad_sizes(P.C)[1]:
        for Kc in (KC_SIZES if M < 200 else (1, 9, 129)):
            rng = np.random.default_rng([M, Kc, 2])
            _, _, H = ref.hessian(rng, 2 * M, M)
            S = np.linalg.inv(H); S = (S + S.T) / 2
            G = rng.normal(size=(M, Kc)); v = rng.normal(size=M)
            q, l = run_quad(P, G, S, v, rng)
            rq, rl = ref.quad_ref(G, S, v)
            qb, lb = ref.quad_bound(G, S, v)
            r = max(ref.ratio(np.abs(q - rq).astype(np.float64), qb), ref.ratio(np.abs(l - rl).astype(np.float64), lb))
            worst = max(worst, (r, (M, Kc)))
            assert r <= 1.0, f"quad_forms_mma M={M} Kc={Kc}: worst error/bound {r:.3g}"
    print(f"quad_forms_mma: worst error/bound {worst[0]:.3g} at (M, Kc) = {worst[1]}")


@pytest.mark.parametrize("kind", ["simt", "mma"])
def test_quad_invariants(P, kind):
    """Duplicates tie bitwise; outputs follow a candidate permutation; the physical row order changes nothing."""
    T = P.C["FIT_T"]
    for M in quad_sizes(P.C)[0 if kind == "simt" else 1]:
        Kc = 1100
        rng = np.random.default_rng([M, 3])
        _, _, H = ref.hessian(rng, 2 * M, M)
        S = np.linalg.inv(H); S = (S + S.T) / 2
        G = rng.normal(size=(M, Kc)); v = rng.normal(size=M)
        dups = _dups(Kc, T)
        G[:, dups] = G[:, [3]]
        q, l = run_quad(P, G, S, v, rng)
        assert bits_equal(q[dups], np.full(len(dups), q[3])) and bits_equal(l[dups], np.full(len(dups), l[3])), \
            f"quad_forms_{kind} M={M}: duplicates at {dups} do not tie: {q[dups]}"
        perm = rng.permutation(Kc)
        qp, lp = run_quad(P, G[:, perm], S, v, rng)
        assert bits_equal(qp, q[perm]) and bits_equal(lp, l[perm]), f"quad_forms_{kind} M={M}: outputs do not follow a permutation"
        grow = rng.permutation(M + 40)[:M].astype(np.int32)
        qg, lg = run_quad(P, G, S, v, grow=grow)
        assert bits_equal(qg, q) and bits_equal(lg, l), f"quad_forms_{kind} M={M}: outputs depend on the physical row order"


# ---------------------------------------------------------------------------------------------------------------------
# gram_pipe / gram_mma

GRAM_N = (1, 2, 31, 32, 33, 63, 64, 65, 1001)


def gram_pipe_M(C):
    return sorted({1, 4, 5, 31, 32, 33, C["PHIT_LD"] - 1, C["PHIT_LD"]})


def gram_mma_M(C):
    p = C["PHIT_LD"]
    return [p + 1, p + 8, p + 9, p + 16, 2 * p + 1, 200]


def test_gram_pipe_bitwise(P):
    """gram_pipe (H and the gradient PHI'ev) against the C restatement on realistic inputs, and exact on exact ones."""
    for M in gram_pipe_M(P.C):
        for N in GRAM_N:
            rng = np.random.default_rng([N, M])
            phi, w, _ = ref.hessian(rng, N, M)
            ev = rng.normal(size=N)
            H, g = run_gram(P, phi, w, ev)
            cH, cg = ref.c_gram_pipe(phi, w, ev, P.C["FIT_T"])
            iu = np.triu_indices(M)
            assert bits_equal(H[iu], cH[iu]), f"gram_pipe N={N} M={M}: {np.count_nonzero(H[iu] != cH[iu])} entries differ from C"
            assert bits_equal(g, cg), f"gram_pipe N={N} M={M}: gradient differs from C in {np.count_nonzero(g != cg)} entries"
            H1, _ = run_gram(P, phi)                                   # w = null: all ones
            cH1, _ = ref.c_gram_pipe(phi, None, None, P.C["FIT_T"])
            assert bits_equal(H1[iu], cH1[iu]), f"gram_pipe N={N} M={M}, w = 1: differs from C"
            phi = ref.int_cache(rng, M, N, -2, 2); w = np.ldexp(rng.integers(1, 17, N).astype(np.float64), -6); ev = ref.dyadic(rng, N)
            assert ref.gram_certificate(phi, w, ev)
            H, g = run_gram(P, phi, w, ev)
            E = (phi * w) @ phi.T
            assert np.array_equal(H[iu], E[iu]) and np.array_equal(g, phi @ ev), f"gram_pipe N={N} M={M}: not exact on an exact case"


def test_gram_mma(P):
    """gram_mma: exact on exact cases, within (N + 4) u sum |fl(phi_j w)| |phi_k| on realistic ones."""
    worst = (0.0, (0, 0))
    for M in gram_mma_M(P.C):
        for N in GRAM_N:
            rng = np.random.default_rng([N, M, 5])
            phi = ref.int_cache(rng, M, N, -2, 2); w = np.ldexp(rng.integers(1, 17, N).astype(np.float64), -6)
            assert ref.gram_certificate(phi, w)
            H, _ = run_gram(P, phi, w, mma=True)
            E = (phi * w) @ phi.T
            iu = np.triu_indices(M)
            assert np.array_equal(H[iu], E[iu]), f"gram_mma N={N} M={M}: {np.count_nonzero(H[iu] != E[iu])} entries not exact"
            if N in (1, 33, 65, 1001):
                phi, w, _ = ref.hessian(rng, N, M)
                H, _ = run_gram(P, phi, w, mma=True)
                hi, lo = ref.gram_ref(phi, w)
                r = ref.ratio(np.abs((H - hi) - lo)[iu], ref.gram_bound(phi, w)[iu])
                worst = max(worst, (r, (N, M)))
                assert r <= 1.0, f"gram_mma N={N} M={M}: worst error/bound {r:.3g}"
    print(f"gram_mma: worst error/bound {worst[0]:.3g} at (N, M) = {worst[1]}")


# ---------------------------------------------------------------------------------------------------------------------
# cache_dot, sym_matvec_row

def test_cache_dot_bitwise(P):
    T = P.C["FIT_T"]
    for M in (1, 3, 4, 5, 63, 64, 65, ROWOFF_M + 1):
        for Kc in (1, T - 1, T, T + 1, 2 * T - 1, 2 * T, 2 * T + 1, 1100):
            rng = np.random.default_rng([M, Kc, 6])
            G = rng.normal(size=(M, Kc)); vec = rng.normal(size=M)
            z = run_cache_dot(P, G, vec, rng)
            cz = ref.c_cache_dot(G, vec)
            assert bits_equal(z, cz), f"cache_dot M={M} Kc={Kc}: {np.count_nonzero(z != cz)} differ from C"
            perm = rng.permutation(Kc)
            assert bits_equal(run_cache_dot(P, G[:, perm], vec, rng), z[perm]), f"cache_dot M={M} Kc={Kc}: permutation"


def test_sym_matvec_bitwise(P):
    for M in (1, 2, 3, 4, 5, 7, 8, 9, 64, 65, 633, BASIS_CAP):
        rng = np.random.default_rng([M, 7])
        A = rng.normal(size=(M, M)); A = (A + A.T) / 2; v = rng.normal(size=M)
        z = run_sym_matvec(P, A, v)
        cz = ref.c_sym_matvec(A, v)
        assert bits_equal(z, cz), f"sym_matvec_row M={M}: {np.count_nonzero(z != cz)} differ from C"
