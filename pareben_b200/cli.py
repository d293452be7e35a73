"""R-free command line around the hot path:  python -m pareben_b200.cli <command> ...

  cv          CrossValidate(BASIS, Target, nFolds, Epis, prior, search) from files -> optimum + Results.Summary (TSV/JSON)
  cv-multi    CrossValidateMulti: several responses of one design (--target repeated, or one .npy/.npz n x T matrix)
              in one call -> a JSON list with one `cv` object per response
  fit         EBelasticNet.Gaussian / .Binomial at given (lambda, alpha) -> the weight table
  lambda-max  GetLambdaMax
  sl-filter   the single-locus prefilter of SL_filter.R

Inputs: genotype text (optionally zipped) + phenotype text as in the reference's scripts
(paper_materials/Real Data Analysis/Full_Test/dataprep.R:3-4, Timing Tests/test_time_Gaus.R:13-19), or .rda / .RDS /
.npy / .npz matrices.  Everything numeric runs in libpareben.so on the GPU(s); there is no CPU path."""
from __future__ import annotations

import argparse
import json
import sys
import time

import numpy as np

from . import cross_validate as cv
from . import io as pio


def _common(sp):
    sp.add_argument("--basis", required=True, help="genotype text (.txt/.tsv/.zip) or matrix (.rda/.RDS/.npy/.npz)")
    sp.add_argument("--target", required=True, help="phenotype text (id value) or vector file")
    sp.add_argument("--basis-name", default=None); sp.add_argument("--target-name", default=None)
    sp.add_argument("--epis", default="no", choices=["no", "yes"])
    sp.add_argument("--prior", default="gaussian", choices=["gaussian", "binomial"])
    sp.add_argument("--rows", type=int, default=0, help="use only the first ROWS rows"); sp.add_argument("--cols", type=int, default=0)
    sp.add_argument("--device", type=int, default=None)
    sp.add_argument("--out", default="-", help="output file (default stdout)")


def _load(a):
    t = time.perf_counter()
    X, y = pio.load_problem(a.basis, a.target, a.basis_name, a.target_name)
    if a.rows:
        X, y = X[:a.rows], y[:a.rows]
    if a.cols:
        X = X[:, :a.cols]
    print(f"[pareben] loaded BASIS {X.shape[0]} x {X.shape[1]} ({X.dtype}), Target {y.size} in {time.perf_counter() - t:.2f} s", file=sys.stderr)
    return X, y


def _cv_out(a, r):
    """The `cv` command's JSON object for one CrossValidate result."""
    if a.search == "global":
        key = "MSE" if a.prior == "gaussian" else "Likelihood"
        return {"lambda.optimal": float(r["lambda.optimal"]), "alpha.optimal": float(r["alpha.optimal"]),
                "Results.Summary": {c: np.asarray(r["Results.Summary"][c]).tolist() for c in ("alpha", "lambda", "SE", key)}}
    return {"lambda.optimal": float(r["lambda.optimal"]), "alpha.optimal": float(r["alpha.optimal"]),
            "CrossValidation": np.asarray(r["CrossValidation"]).tolist()}


def _cv_multi(a):
    t = time.perf_counter()
    X, Y = pio.load_problem_multi(a.basis, a.target, a.basis_name, a.target_name)
    if a.rows:
        X, Y = X[:a.rows], Y[:a.rows]
    if a.cols:
        X = X[:, :a.cols]
    print(f"[pareben] loaded BASIS {X.shape[0]} x {X.shape[1]} ({X.dtype}), Targets {Y.shape[0]} x {Y.shape[1]} in "
          f"{time.perf_counter() - t:.2f} s", file=sys.stderr)
    t = time.perf_counter()
    folds = cv.AssignToFolds(X, a.nfolds, sample_kind=a.sample_kind)
    rs = cv.CrossValidateMulti(X, Y, a.nfolds, folds, a.epis, a.prior, a.search, device=a.device, sample_kind=a.sample_kind,
                               n_devices=a.devices)
    print(f"[pareben] {Y.shape[1]} responses cross-validated in {time.perf_counter() - t:.2f} s", file=sys.stderr)
    _emit(a, [_cv_out(a, r) for r in rs])
    return 0


def _emit(a, obj):
    text = json.dumps(obj, indent=1)
    if a.out == "-":
        print(text)
    else:
        open(a.out, "w").write(text + "\n")


def main(argv=None):
    ap = argparse.ArgumentParser(prog="pareben", description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    sub = ap.add_subparsers(dest="cmd", required=True)
    s = sub.add_parser("cv"); _common(s)
    s.add_argument("--nfolds", type=int, required=True); s.add_argument("--search", default="global", choices=["global", "local"])
    s.add_argument("--devices", type=int, default=1, help="GPUs sharing the grid (0 = all visible)")
    s.add_argument("--sample-kind", default="Rejection", choices=["Rejection", "Rounding"], help="R's sample.kind for AssignToFolds")
    s = sub.add_parser("cv-multi")
    s.add_argument("--basis", required=True, help="genotype text (.txt/.tsv/.zip) or matrix (.rda/.RDS/.npy/.npz)")
    s.add_argument("--target", required=True, action="append",
                   help="one response: phenotype text (id value) or vector file; repeat for more.  Or one .npy/.npz n x T matrix")
    s.add_argument("--basis-name", default=None); s.add_argument("--target-name", default=None)
    s.add_argument("--epis", default="no", choices=["no", "yes"])
    s.add_argument("--prior", default="gaussian", choices=["gaussian", "binomial"])
    s.add_argument("--rows", type=int, default=0, help="use only the first ROWS rows"); s.add_argument("--cols", type=int, default=0)
    s.add_argument("--device", type=int, default=None)
    s.add_argument("--out", default="-", help="output file (default stdout)")
    s.add_argument("--nfolds", type=int, required=True); s.add_argument("--search", default="global", choices=["global", "local"])
    s.add_argument("--devices", type=int, default=1, help="GPUs sharing the grid (0 = all visible)")
    s.add_argument("--sample-kind", default="Rejection", choices=["Rejection", "Rounding"], help="R's sample.kind for AssignToFolds")
    s = sub.add_parser("fit"); _common(s)
    s.add_argument("--lambda", dest="lam", type=float, required=True); s.add_argument("--alpha", type=float, required=True)
    s = sub.add_parser("lambda-max"); _common(s)
    s = sub.add_parser("sl-filter"); _common(s)
    s.add_argument("--tau-main", type=float, default=0.02); s.add_argument("--tau-pair", type=float, default=0.05)
    a = ap.parse_args(argv)
    if a.cmd == "cv-multi":
        return _cv_multi(a)
    X, y = _load(a)
    t = time.perf_counter()
    if a.cmd == "cv":
        folds = cv.AssignToFolds(X, a.nfolds, sample_kind=a.sample_kind)
        if a.search == "global":
            r = cv.CrossValidate(X, y, a.nfolds, folds, a.epis, a.prior, "global", device=a.device, n_devices=a.devices)
        else:
            r = cv.LocalSearch(X, y, a.nfolds, a.epis, folds, a.prior, device=a.device)
        out = _cv_out(a, r)
    elif a.cmd == "fit":
        f = (cv.EBelasticNet_Gaussian if a.prior == "gaussian" else cv.EBelasticNet_Binomial)(X, y, a.lam, a.alpha, a.epis, device=a.device)
        out = {k: (np.asarray(v).tolist() if isinstance(v, np.ndarray) else v) for k, v in f.items()}
    elif a.cmd == "lambda-max":
        out = {"lambda_max": cv.GetLambdaMax(X, y, a.epis, device=a.device)}
    else:
        r = cv.SLFilter(X, y, a.tau_main, a.tau_pair, a.epis, device=a.device)
        out = {k: np.asarray(v).tolist() for k, v in r.items()}
    out["seconds"] = time.perf_counter() - t
    _emit(a, out)
    return 0


if __name__ == "__main__":
    sys.exit(main())
