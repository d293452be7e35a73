"""Test helper: a compact pareben_fit_batch record expanded into the reference-layout table pareben_fit returns
(include/pareben.h): Gaussian main k x 4 and Gaussian Epis k(k+1)/2 x 5 indexed by candidate id, binomial main k x 4
indexed by column id, binomial Epis 2k x 4 compact in Used order with decoded loci.  The tests compare tables built here
with pareben_fit's own, and _weight_table of these tables with the weight tables EBelasticNetMulti builds."""
import numpy as np

from pareben_b200.cross_validate import candidate_loci


def expand(n_effects, cand, beta, var, k, epis, gaussian):
    m = int(n_effects)
    c = np.asarray(cand[:m], dtype=np.int64) - 1
    if gaussian:
        kc = (k + 1) * k // 2 if epis else k
        table = np.zeros((kc, 5 if epis else 4))
        li, lj = candidate_loci(np.arange(kc), k)
        table[:, 0], table[:, 1] = li, lj
        table[c, 2], table[c, 3] = beta[:m], var[:m]
        if epis:
            table[c, 4] = c + 1
        return table
    if not epis:
        table = np.zeros((k, 4))
        table[:, 0] = table[:, 1] = np.arange(1, k + 1)
        table[c, 2], table[c, 3] = beta[:m], var[:m]
        return table
    table = np.zeros((2 * k, 4))
    r = min(m, 2 * k)
    li, lj = candidate_loci(c[:r], k)
    table[:r, 0], table[:r, 1], table[:r, 2], table[:r, 3] = li, lj, beta[:r], var[:r]
    return table


def keep_rows(table, epis, gaussian):
    """The rows EBelasticNet_Gaussian / _Binomial hand to _weight_table."""
    return np.nonzero(table[:, 4] != 0)[0] if (gaussian and epis) else np.nonzero(table[:, 2] != 0)[0]
