/* pareben_call.c -- the `.Call` shim an R package maintainer adds under parEBEN/src/.
 * Thin by design: it only converts SEXPs to the plain pointers of include/pareben.h.
 * Build inside the R package with  PKG_LIBS = -L<dir of libpareben.so> -lpareben
 * (cannot be compiled in the build container: R headers are absent; the C-ABI it calls is
 * exercised from Python in tests/).
 *
 * Entry points (all registered below):
 *   pareben_cv_grid_call     CrossValidate / LocalSearch: the whole (alpha, lambda) x fold table, nDevices GPUs
 *   pareben_cv_grid_multi_call  the same for the T columns of a response matrix against one BASIS, in one call
 *   pareben_lambda_max_call  GetLambdaMax (R/BuildGrid.R:5-32), incl. the K^2/2 pair scan of Epis = "yes"
 *   pareben_fit_call         EBelasticNet.Gaussian / .Binomial: the `.C` outputs of one all-rows fit
 *   pareben_sl_filter_call   the single-locus prefilter of SL_filter.R
 * EBEN's own `.C` symbols (elasticNetLinearNeMainEff, ...) are exported by libpareben.so itself under their original
 * names: EBEN's R wrappers need no shim at all, only `useDynLib(pareben)`. */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include "pareben.h"

static void dims(SEXP BASIS, int *n, int *k)
{
    SEXP dim = getAttrib(BASIS, R_DimSymbol);
    if (!isReal(BASIS) || isNull(dim) || LENGTH(dim) != 2) error("BASIS must be a double matrix");
    *n = INTEGER(dim)[0]; *k = INTEGER(dim)[1];
}

static SEXP named_list(int n, const char **names, SEXP *items)
{
    SEXP out = PROTECT(allocVector(VECSXP, n)), nm = PROTECT(allocVector(STRSXP, n));
    for (int i = 0; i < n; i++) { SET_VECTOR_ELT(out, i, items[i]); SET_STRING_ELT(nm, i, mkChar(names[i])); }
    setAttrib(out, R_NamesSymbol, nm);
    UNPROTECT(2);
    return out;
}

/* .Call("pareben_cv_grid_call", BASIS, Target, foldId, nFolds, alpha, lambda, epis, prior, nDevices, device)
 * nDevices GPUs starting at `device` share the grid (0 = every visible GPU): the in-library replacement of the
 * foreach fan-out over registered workers (R/CrossValidate.R:66-70).
 * returns list(fold_err = matrix[nFolds x nGrid], status = integer matrix, n_selected = integer matrix);
 * column g of fold_err holds the nFolds hold-out errors of grid row g, so as.vector(fold_err)
 * is already in Results.Detail order (grid row major, fold minor). */
SEXP pareben_cv_grid_call(SEXP BASIS, SEXP Target, SEXP foldId, SEXP nFolds, SEXP alpha, SEXP lambda,
                          SEXP epis, SEXP prior, SEXP nDevices, SEXP device)
{
    int n, k;
    dims(BASIS, &n, &k);
    const int nf = asInteger(nFolds), ng = LENGTH(alpha);
    if (LENGTH(Target) != n || LENGTH(foldId) != n || LENGTH(lambda) != ng) error("argument lengths disagree");
    SEXP err = PROTECT(allocMatrix(REALSXP, nf, ng));
    SEXP st = PROTECT(allocMatrix(INTSXP, nf, ng));
    SEXP ns = PROTECT(allocMatrix(INTSXP, nf, ng));
    const int rc = pareben_cv_grid(REAL(BASIS), n, k, REAL(Target), INTEGER(foldId), nf, REAL(alpha), REAL(lambda),
                                   ng, asInteger(epis), asInteger(prior), asInteger(nDevices), asInteger(device), 0, 1,
                                   REAL(err), INTEGER(st), INTEGER(ns));
    if (rc != PAREBEN_OK) { UNPROTECT(3); error("pareben_cv_grid failed (%d): %s", rc, pareben_last_error()); }
    const char *names[] = {"fold_err", "status", "n_selected"};
    SEXP items[] = {err, st, ns};
    SEXP out = named_list(3, names, items);
    UNPROTECT(3);
    return out;
}

/* .Call("pareben_cv_grid_multi_call", BASIS, Targets, foldId, nFolds, alpha, lambda, epis, prior, nDevices, device)
 * Targets: n x T double matrix, one response per column (traits of one design, permuted copies of one response).
 * alpha, lambda: nGrid x T matrices, column t = the grid of response t (its own BuildGrid / GetLambdaMax).
 * returns list(fold_err = array[nFolds x nGrid x T], status, n_selected): slice [, , t] is what pareben_cv_grid_call
 * returns for Targets[, t] alone, bitwise (pareben_cv_grid_multi's table order, fold fastest). */
SEXP pareben_cv_grid_multi_call(SEXP BASIS, SEXP Targets, SEXP foldId, SEXP nFolds, SEXP alpha, SEXP lambda,
                                SEXP epis, SEXP prior, SEXP nDevices, SEXP device)
{
    int n, k, nt, ng;
    dims(BASIS, &n, &k);
    dims(Targets, &nt, &ng);          /* rows, responses */
    if (nt != n) error("Targets must have nrow(BASIS) rows");
    const int T = ng, nf = asInteger(nFolds);
    if (T < 1 || LENGTH(alpha) % T != 0) error("alpha must be an nGrid x ncol(Targets) matrix");
    ng = LENGTH(alpha) / T;
    if (ng < 1 || LENGTH(foldId) != n || LENGTH(lambda) != LENGTH(alpha)) error("argument lengths disagree");
    SEXP dim = PROTECT(allocVector(INTSXP, 3));
    INTEGER(dim)[0] = nf; INTEGER(dim)[1] = ng; INTEGER(dim)[2] = T;
    SEXP err = PROTECT(allocArray(REALSXP, dim)), st = PROTECT(allocArray(INTSXP, dim)), ns = PROTECT(allocArray(INTSXP, dim));
    const int rc = pareben_cv_grid_multi(REAL(BASIS), n, k, REAL(Targets), T, INTEGER(foldId), nf, REAL(alpha), REAL(lambda), ng,
                                         asInteger(epis), asInteger(prior), asInteger(nDevices), asInteger(device), 0, 1,
                                         REAL(err), INTEGER(st), INTEGER(ns));
    if (rc != PAREBEN_OK) { UNPROTECT(4); error("pareben_cv_grid_multi failed (%d): %s", rc, pareben_last_error()); }
    const char *names[] = {"fold_err", "status", "n_selected"};
    SEXP items[] = {err, st, ns};
    SEXP out = named_list(3, names, items);
    UNPROTECT(4);
    return out;
}

/* .Call("pareben_lambda_max_call", BASIS, Target, epis, device) -> numeric(1): GetLambdaMax before the x10 */
SEXP pareben_lambda_max_call(SEXP BASIS, SEXP Target, SEXP epis, SEXP device)
{
    int n, k;
    dims(BASIS, &n, &k);
    if (LENGTH(Target) != n) error("argument lengths disagree");
    pareben_problem *p = NULL;
    double lm = 0;
    int rc = pareben_problem_create(&p, asInteger(device), REAL(BASIS), n, k, REAL(Target), NULL, 0, asInteger(epis), PAREBEN_GAUSSIAN);
    if (rc == PAREBEN_OK) rc = pareben_lambda_max(p, &lm);
    if (p) pareben_problem_destroy(p);
    if (rc != PAREBEN_OK) error("pareben_lambda_max failed (%d): %s", rc, pareben_last_error());
    return ScalarReal(lm);
}

/* .Call("pareben_fit_call", BASIS, Target, lambda, alpha, epis, prior, device)
 * -> list(Beta = matrix in the `.C` layout, WaldScore, Intercept, extra = residual variance | logLikelihood, status):
 * what `.C("elasticNetLinearNeMainEff", ...)` etc. return (EBelasticNet.Gaussian.R:39-51, .Binomial.R:33-46). */
SEXP pareben_fit_call(SEXP BASIS, SEXP Target, SEXP lambda, SEXP alpha, SEXP epis, SEXP prior, SEXP device)
{
    int n, k;
    dims(BASIS, &n, &k);
    if (LENGTH(Target) != n) error("argument lengths disagree");
    const int ep = asInteger(epis), pr = asInteger(prior);
    const double kc = ep ? 0.5 * k * (k + 1.0) : k;
    const int rows = pr == PAREBEN_GAUSSIAN ? (int)kc : (ep ? 2 * k : k), cols = (pr == PAREBEN_GAUSSIAN && ep) ? 5 : 4;
    SEXP beta = PROTECT(allocMatrix(REALSXP, rows, cols));
    SEXP wald = PROTECT(allocVector(REALSXP, 1)), icpt = PROTECT(allocVector(REALSXP, pr == PAREBEN_GAUSSIAN ? 1 : 2));
    SEXP extra = PROTECT(allocVector(REALSXP, 1)), st = PROTECT(allocVector(INTSXP, 1));
    pareben_problem *p = NULL;
    int rc = pareben_problem_create(&p, asInteger(device), REAL(BASIS), n, k, REAL(Target), NULL, 0, ep, pr);
    if (rc == PAREBEN_OK) rc = pareben_fit(p, asReal(alpha), asReal(lambda), REAL(beta), REAL(wald), REAL(icpt), REAL(extra), INTEGER(st));
    if (p) pareben_problem_destroy(p);
    if (rc != PAREBEN_OK) { UNPROTECT(5); error("pareben_fit failed (%d): %s", rc, pareben_last_error()); }
    const char *names[] = {"Beta", "WaldScore", "Intercept", "extra", "status"};
    SEXP items[] = {beta, wald, icpt, extra, st};
    SEXP out = named_list(5, names, items);
    UNPROTECT(5);
    return out;
}

/* .Call("pareben_sl_filter_call", BASIS, Target, tauMain, tauPair, epis, device)
 * -> list(cand = 0-based candidate ids ascending (0..k-1 main effects, then pairs i < j row-major), stat) */
SEXP pareben_sl_filter_call(SEXP BASIS, SEXP Target, SEXP tauMain, SEXP tauPair, SEXP epis, SEXP device)
{
    int n, k;
    dims(BASIS, &n, &k);
    if (LENGTH(Target) != n) error("argument lengths disagree");
    pareben_problem *p = NULL;
    int rc = pareben_problem_create(&p, asInteger(device), REAL(BASIS), n, k, REAL(Target), NULL, 0, asInteger(epis), PAREBEN_GAUSSIAN);
    int kept = 0;
    if (rc == PAREBEN_OK) rc = pareben_sl_filter(p, asReal(tauMain), asReal(tauPair), 0, NULL, NULL, &kept);   /* count */
    SEXP cand = PROTECT(allocVector(INTSXP, kept)), stat = PROTECT(allocVector(REALSXP, kept));
    if (rc == PAREBEN_OK && kept > 0) rc = pareben_sl_filter(p, asReal(tauMain), asReal(tauPair), kept, INTEGER(cand), REAL(stat), &kept);
    if (p) pareben_problem_destroy(p);
    if (rc != PAREBEN_OK) { UNPROTECT(2); error("pareben_sl_filter failed (%d): %s", rc, pareben_last_error()); }
    const char *names[] = {"cand", "stat"};
    SEXP items[] = {cand, stat};
    SEXP out = named_list(2, names, items);
    UNPROTECT(2);
    return out;
}

static const R_CallMethodDef call_methods[] = {
    {"pareben_cv_grid_call", (DL_FUNC)&pareben_cv_grid_call, 10},
    {"pareben_cv_grid_multi_call", (DL_FUNC)&pareben_cv_grid_multi_call, 10},
    {"pareben_lambda_max_call", (DL_FUNC)&pareben_lambda_max_call, 4},
    {"pareben_fit_call", (DL_FUNC)&pareben_fit_call, 7},
    {"pareben_sl_filter_call", (DL_FUNC)&pareben_sl_filter_call, 6},
    {NULL, NULL, 0}
};

void R_init_parEBEN(DllInfo *dll)
{
    R_registerRoutines(dll, NULL, call_methods, NULL, NULL);
    R_useDynamicSymbols(dll, FALSE);
}
