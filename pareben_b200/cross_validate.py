"""Host-side mirror of parEBEN's R interface, driving the CUDA library through its C-ABI.

Same names, argument meaning and return shapes as the reference (R is not available in this
image, so this Python layer stands where R/CrossValidate.R etc. would call `.Call`):
  CrossValidate   /root/reference/R/CrossValidate.R:61-117
  BuildGrid       /root/reference/R/BuildGrid.R:34-52     GetLambdaMax  :5-32
  AssignToFolds   /root/reference/R/AssignToFolds.R:6-19
  LocalSearch     /root/reference/R/LocalSearch.R:6-130
  CrossValidateMulti  (no reference counterpart: the reference loops CrossValidate) T responses against one design in
                  one upload and one batched fit call, each result equal to CrossValidate on that response
  EBelasticNet_Gaussian / EBelasticNet_Binomial  (final model after CV, README.md:89-94;
                  /root/reference/EBEN_orig/R/EBelasticNet.Gaussian.R, .Binomial.R)
The foreach/%dopar% fan-out (CrossValidate.R:66-70, 88-92; LocalSearch.R:67-104) is replaced
by ONE batched launch per GPU; with torch.distributed initialised (one process per GPU) the
fits are sharded by cost-aware interleaving and merged with one tiny all-reduce.

Documented deviations from the reference as written (SURVEY.md facts 3, 4):
  * prior="binomial", search="global": the reference selects with which.min(Error$MSE) on a
    table that has no MSE column and returns empty optima; here the intended rule
    which.min(Likelihood) (Likelihood = -mean logL) is used.
  * prior="binomial", search="local": the reference prints a message and fails on an undefined
    variable; here the same early-stopping walk is applied to Likelihood.
"""
from __future__ import annotations

import math

import numpy as np

from . import _lib, rcompat


def _as_matrix(BASIS):
    X = np.asarray(BASIS, dtype=np.float64)
    if X.ndim != 2:
        raise ValueError("BASIS must be a matrix")
    return X


def GetLambdaMax(BASIS, Target, Epis="no", device: int | None = None) -> float:
    """GetLambdaMax (BuildGrid.R:5-32) on the device; the Epis pair scan (K^2/2 columns generated on
    the fly) is the part that is quadratic in K."""
    with _lib.Problem(_as_matrix(BASIS), Target, None, 0, Epis == "yes", "gaussian", device) as p:
        return p.lambda_max()


def _grid_from_lambda_max(lam_max: float):
    """The 20 x 20 grid of BuildGrid.R:36-51 from GetLambdaMax's value: expand.grid order (alpha fastest)."""
    lam_max = lam_max * 10
    lam_min = math.log(0.001 * lam_max)
    step = (math.log(lam_max) - lam_min) / 19
    Lambda = np.exp(rcompat.seq(math.log(lam_max), lam_min, -step))
    Alpha = rcompat.seq(1.0, 0.05, -0.05)
    return {"alpha": np.tile(Alpha, Lambda.size), "lambda": np.repeat(Lambda, Alpha.size)}


def BuildGrid(BASIS, Target, nFolds=0, Epis="no", device: int | None = None):
    """BuildGrid (BuildGrid.R:34-52) -> dict(alpha=[400], lambda=[400]) in expand.grid order (alpha fastest)."""
    return _grid_from_lambda_max(GetLambdaMax(BASIS, Target, Epis, device))


def AssignToFolds(BASIS, nFolds=0, foldId=0, sample_kind: str = "Rejection", rng: rcompat.RRandom | None = None):
    """AssignToFolds (AssignToFolds.R:6-19): set.seed(1), then a balanced random labelling."""
    N = _as_matrix(BASIS).shape[0]
    rng = rng or rcompat.RRandom(1, sample_kind)
    if np.size(foldId) != N:
        labels = list(np.tile(np.arange(1, nFolds + 1), N // nFolds))
        if N % nFolds != 0:
            labels += list(range(1, N % nFolds + 1))
        foldId = rng.sample(labels)
    return np.asarray(foldId, dtype=np.int32)


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            return dist
    except Exception:
        pass
    return None


def _merge_shards(err, st, ns, device):
    """The `.combine = rbind` of the reference across ranks: every rank filled only its own entries (the rest are 0),
    so one all-reduce(sum) of the three small tables is the gather.  No-op without an initialised process group."""
    dist = _dist()
    if dist is None:
        return err, st, ns
    import torch
    on_gpu = dist.get_backend() == "nccl"
    dev = torch.device("cuda", _lib.default_device() if device is None else device) if on_gpu else torch.device("cpu")
    packed = torch.from_numpy(np.concatenate([err.ravel(), st.ravel().astype(np.float64), ns.ravel().astype(np.float64)])).to(dev)
    dist.all_reduce(packed)
    packed = packed.cpu().numpy()
    m = err.size
    return (packed[:m].reshape(err.shape), packed[m:2 * m].astype(np.int32).reshape(err.shape),
            packed[2 * m:].astype(np.int32).reshape(err.shape))


def _grid_and_errors(X, y, fold_id, n_folds, Epis, prior, device, n_devices=1):
    """BuildGrid + all n_grid x n_folds hold-out errors.  One process, one GPU: BASIS is uploaded ONCE and the same
    resident problem serves GetLambdaMax and the fits.  n_devices != 1: one call fans the grid over that many GPUs of
    this process (pareben_cv_grid's worker threads).  With torch.distributed up (one process per GPU) every rank
    computes its shard and the shards are merged by _merge_shards."""
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    epis = Epis == "yes"
    if n_devices != 1:
        grid = BuildGrid(X, y, n_folds, Epis, device)
        err, st, ns = _lib.cv_grid(X, y, fold_id, n_folds, grid["alpha"], grid["lambda"], epis, prior, device, rank, world, n_devices)
    else:
        with _lib.Problem(X, y, fold_id, n_folds, epis, prior, device) as p:
            grid = _grid_from_lambda_max(p.lambda_max())
            err, st, ns = p.cv_grid(grid["alpha"], grid["lambda"], rank, world)
    err, st, ns = _merge_shards(err, st, ns, device)
    return grid, err, st, ns


def _which_min(values, status, what):
    """R's which.min: first minimum, NA skipped.  A table that is all NA stops, as the reference does on
    is.na(Mu0); fits that ended with a non-zero status are reported (the reference prints and carries on)."""
    bad = np.asarray(status) != 0
    if bad.any():
        import warnings
        st = np.asarray(status)
        warnings.warn(f"{int(bad.sum())} of {st.size} fits finished with a non-zero status "
                      f"(basis cap {int((st & _lib.FIT_BASIS_CAP > 0).sum())}, not positive definite {int((st & _lib.FIT_NOT_PD > 0).sum())}, "
                      f"non-finite {int((st & _lib.FIT_NONFINITE > 0).sum())}, iteration limit {int((st & _lib.FIT_ITER_MAX > 0).sum())})",
                      RuntimeWarning, stacklevel=3)
    values = np.asarray(values, dtype=np.float64)
    if np.all(np.isnan(values)):
        raise ValueError(f"every {what} is NA: no optimum can be selected")
    return int(np.nanargmin(values))


def _summarise(alpha, lam, fold_err, value_name):
    """group_by(alpha, lambda) %>% summarise(SE = sd/sqrt(nFolds), mean)  (CrossValidate.R:72-76, 93-97):
    rows sorted by alpha then lambda ascending."""
    order = np.lexsort((lam, alpha))
    n_folds = fold_err.shape[1]
    se = np.array([rcompat.sd(fold_err[r]) / math.sqrt(n_folds) for r in order])
    mean = np.array([rcompat.mean(fold_err[r]) for r in order])
    return {"alpha": alpha[order], "lambda": lam[order], "SE": se,
            value_name: mean if value_name == "MSE" else -mean}


def CrossValidate(BASIS, Target, nFolds, foldId=0, Epis="no", prior="gaussian", search="global",
                  device: int | None = None, sample_kind: str = "Rejection", n_devices: int = 1):
    """CrossValidate (CrossValidate.R:61-117).  Returns a dict with the reference's four entries.
    device: GPU of this process (default LOCAL_RANK, else 0); n_devices: GPUs this ONE call fans the grid over."""
    X = _as_matrix(BASIS)
    y = np.asarray(Target, dtype=np.float64).ravel()
    prior_key = "gaussian" if prior == "gaussian" else "binomial"     # anything else = binomial branch (:65,87)
    if search != "global":
        return LocalSearch(X, y, nFolds, Epis, foldId, prior, device=device, sample_kind=sample_kind, n_devices=n_devices)
    # TestModel ignores the caller's foldId and recomputes folds with set.seed(1) (TestModel.R:9)
    folds = AssignToFolds(X, nFolds, sample_kind=sample_kind)
    grid, err, status, nsel = _grid_and_errors(X, y, folds, nFolds, Epis, prior_key, device, n_devices)
    return _global_result(grid, err, status, nsel, folds, nFolds, prior_key)


def _global_result(grid, err, status, nsel, folds, nFolds, prior_key):
    """CrossValidate's return value (CrossValidate.R:72-117) from the grid and its n_grid x n_folds tables."""
    n_grid = grid["alpha"].size
    value = "MSE" if prior_key == "gaussian" else "logL"
    detail = {"foldId": np.tile(np.arange(1, nFolds + 1), n_grid), "alpha": np.repeat(grid["alpha"], nFolds),
              "lambda": np.repeat(grid["lambda"], nFolds), value: err.ravel().copy()}
    summary = _summarise(grid["alpha"], grid["lambda"], err, "MSE" if prior_key == "gaussian" else "Likelihood")
    col = "MSE" if prior_key == "gaussian" else "Likelihood"
    idx = _which_min(summary[col], status, col)                                          # which.min (:78, intent of :99)
    return {"Results.Detail": detail, "Results.Summary": summary,
            "lambda.optimal": float(summary["lambda"][idx]), "alpha.optimal": float(summary["alpha"][idx]),
            "status": status, "n_selected": nsel, "foldId": folds}


def LocalSearch(BASIS, Target, nFolds, Epis="no", foldId=0, prior="gaussian", device: int | None = None,
                sample_kind: str = "Rejection", rng: rcompat.RRandom | None = None, n_devices: int = 1):
    """LocalSearch (LocalSearch.R:6-130).  Every fit is independent of visiting order, so the whole
    alpha x lambda x fold table is computed in one batched launch and the early-stopping walk
    (:56-122) is replayed over it; rows the walk never reaches stay zero in fullCV, as in the
    reference.  Folds: the caller's foldId when it has length N, else sample() from the session
    RNG (here: `rng`, default a fresh set.seed(1) stream -- the reference leaves it unseeded)."""
    X = _as_matrix(BASIS)
    y = np.asarray(Target, dtype=np.float64).ravel()
    prior_key = "gaussian" if prior == "gaussian" else "binomial"
    folds = AssignToFolds(X, nFolds, foldId, sample_kind, rng)
    grid, err, status, nsel = _grid_and_errors(X, y, folds, nFolds, Epis, prior_key, device, n_devices)
    return _local_result(grid, err, status, folds, nFolds, prior_key)


def _local_result(grid, err, status, folds, nFolds, prior_key):
    """LocalSearch's early-stopping walk (LocalSearch.R:56-122) replayed over a complete n_grid x n_folds table."""
    if prior_key == "binomial":
        err = -err                       # walk on Likelihood = -logL (documented deviation)
    Alpha, Lambda = grid["alpha"][:20], grid["lambda"][::20]
    n_alpha, n_step = Alpha.size, Lambda.size
    full = np.zeros((n_step * n_alpha, 4))
    each = np.zeros((n_alpha, 4))
    step = 0
    for ia in range(n_alpha):
        sse = np.full((n_step, 2), 1e10)
        for i_s in range(n_step):
            upto = i_s if i_s >= 1 else 1            # SSE1Alpha[1:(i_s-1),1]; 1:0 selects row 1
            mi = int(np.nanargmin(sse[:upto, 0]))    # which.min skips NA; rows not yet visited hold 1e10
            previous = sse[mi, 0] + sse[mi, 1]
            fe = err[i_s * 20 + ia]
            m, se = rcompat.mean(fe), rcompat.sd(fe) / math.sqrt(nFolds)
            sse[i_s] = (m, se)
            full[step] = (Alpha[ia], Lambda[i_s], m, se)
            step += 1
            if m - previous > 0:
                break
        idx = int(np.nanargmin(sse[:, 0]))
        each[ia] = (Alpha[ia], Lambda[idx], sse[idx, 0], sse[idx, 1])
    idx = _which_min(each[:, 2], status, "per-alpha minimum")
    return {"CrossValidation": each, "alpha.optimal": float(each[idx, 0]), "lambda.optimal": float(each[idx, 1]),
            "fullCV": full, "status": status, "foldId": folds}


def _targets(X, Targets):
    Y = np.asarray(Targets, dtype=np.float64)
    if Y.ndim != 2 or Y.shape[0] != X.shape[0] or Y.shape[1] < 1:
        raise ValueError(f"Targets must be an n x T matrix (T >= 1) with n = nrow(BASIS) = {X.shape[0]}; got shape {Y.shape}")
    bad = np.nonzero(~np.isfinite(Y).all(axis=0))[0]
    if bad.size:
        raise ValueError(f"Targets column {int(bad[0])} holds non-finite values (NA/NaN/Inf): per-response missing rows are not "
                         "supported; drop the rows for every response, or run CrossValidate on that response alone")
    return Y


def _grids_and_errors_multi(X, Y, fold_id, n_folds, Epis, prior, device, n_devices=1):
    """_grid_and_errors for the T columns of Y: each response's BuildGrid grid from its own lambda_max (one pass over the
    candidates for all of them) and all T x n_grid x n_folds hold-out errors from one fit call.  Sharding and merging as in
    _grid_and_errors."""
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist is not None else (0, 1)
    epis = Epis == "yes"

    def grids_of(p):
        grids = [_grid_from_lambda_max(float(v)) for v in p.lambda_max_multi()]
        return grids, np.stack([g["alpha"] for g in grids]), np.stack([g["lambda"] for g in grids])

    if n_devices != 1:
        with _lib.Problem(X, Y, None, 0, epis, "gaussian", device) as p:
            grids, A, L = grids_of(p)
        err, st, ns = _lib.cv_grid_multi(X, Y, fold_id, n_folds, A, L, epis, prior, device, rank, world, n_devices)
    else:
        with _lib.Problem(X, Y, fold_id, n_folds, epis, prior, device) as p:
            grids, A, L = grids_of(p)
            err, st, ns = p.cv_grid_multi(A, L, rank, world)
    err, st, ns = _merge_shards(err, st, ns, device)
    return grids, err, st, ns


def CrossValidateMulti(BASIS, Targets, nFolds, foldId=0, Epis="no", prior="gaussian", search="global",
                       device: int | None = None, sample_kind: str = "Rejection", n_devices: int = 1):
    """CrossValidate for each column of Targets (n x T) against the same BASIS, in one problem upload and one fit call.
    Returns a list of T dicts; entry t equals CrossValidate(BASIS, Targets[:, t], nFolds, foldId, Epis, prior, search, ...)
    entry for entry: the folds are the same for every response (AssignToFolds does not look at the response), each
    response gets its own grid from its own lambda_max, and every fit is bitwise the single-response fit.  search="local"
    replays LocalSearch's walk per response over the shared table.  Every response must be observed on every row."""
    X = _as_matrix(BASIS)
    Y = _targets(X, Targets)
    prior_key = "gaussian" if prior == "gaussian" else "binomial"
    if search != "global":
        folds = AssignToFolds(X, nFolds, foldId, sample_kind)
    else:
        folds = AssignToFolds(X, nFolds, sample_kind=sample_kind)
    grids, err, status, nsel = _grids_and_errors_multi(X, Y, folds, nFolds, Epis, prior_key, device, n_devices)
    if search != "global":
        return [_local_result(grids[t], err[t], status[t], folds, nFolds, prior_key) for t in range(Y.shape[1])]
    return [_global_result(grids[t], err[t], status[t], nsel[t], folds, nFolds, prior_key) for t in range(Y.shape[1])]


def _weight_table(table, keep, epis, n):
    ncol = table.shape[1]
    blup = table[keep] if keep.size else np.zeros((1, ncol))
    if epis:
        main = blup[blup[:, 0] == blup[:, 1]]
        pair = blup[blup[:, 0] != blup[:, 1]]
        blup = np.vstack([main[np.argsort(main[:, 0], kind="stable")], pair[np.argsort(pair[:, 0], kind="stable")]])
    blup = blup[:, :4]
    t = np.abs(blup[:, 2]) / (np.sqrt(blup[:, 3]) + 1e-20)
    from scipy.stats import t as student
    p = 2 * (1 - student.cdf(t, df=n - 1))
    return np.column_stack([blup, t, p])


def EBelasticNet_Gaussian(BASIS, Target, lam, alpha, Epis="no", verbose=0, device: int | None = None):
    """EBelasticNet.Gaussian (EBelasticNet.Gaussian.R:1-101) through pareben_fit (batch of 1, all rows)."""
    X = _as_matrix(BASIS)
    epis = Epis == "yes"
    with _lib.Problem(X, Target, None, 0, epis, "gaussian", device) as p:
        table, wald, icpt, resid, status = p.fit(alpha, lam)
    keep = np.nonzero(table[:, 4] != 0)[0] if epis else np.nonzero(table[:, 2] != 0)[0]
    return {"weight": _weight_table(table, keep, epis, X.shape[0]), "WaldScore": wald, "Intercept": float(icpt[0]),
            "residVar": resid, "lambda": lam, "alpha": alpha, "status": status}


def EBelasticNet_Binomial(BASIS, Target, lam, alpha, Epis="no", verbose=0, device: int | None = None):
    """EBelasticNet.Binomial (EBelasticNet.Binomial.R:1-85) through pareben_fit."""
    X = _as_matrix(BASIS)
    epis = Epis == "yes"
    with _lib.Problem(X, Target, None, 0, epis, "binomial", device) as p:
        table, wald, icpt, logl, status = p.fit(alpha, lam)
    keep = np.nonzero(table[:, 2] != 0)[0]
    return {"weight": _weight_table(table, keep, epis, X.shape[0]), "logLikelihood": logl, "WaldScore": wald,
            "Intercept": icpt.copy(), "lambda": lam, "alpha": alpha, "status": status}


def SLFilter(BASIS, Target, tau_main: float = 0.02, tau_pair: float = 0.05, Epis: str = "yes", device: int | None = None):
    """The single-locus prefilter that precedes CrossValidate in the published workflow
    (paper_materials/Real Data Analysis/SL_filter.R:17-52): standardised-correlation screening of the main-effect
    columns (> tau_main) and, for Epis="yes", of all pairwise products (> tau_pair), on the device.
    Returns {"main": 1-based column numbers, "pairs": (n, 2) 1-based locus pairs i < j, "stat_main", "stat_pairs"}."""
    X = np.asarray(BASIS, dtype=np.float64)
    k = X.shape[1]
    with _lib.Problem(X, Target, None, 0, Epis == "yes", "gaussian", device=device) as p:
        cand, stat = p.sl_filter(tau_main, tau_pair)
    main = cand < k
    pc = cand[~main].astype(np.int64) - k
    # invert c = i*(2k-i-1)/2 + (j-i-1) for i < j (the enumeration of elasticNetLinearNeFull2.c:115-134)
    i = np.floor(((2 * k - 1) - np.sqrt((2 * k - 1) ** 2 - 8.0 * pc)) / 2).astype(np.int64)
    i = np.where(i * (2 * k - i - 1) // 2 > pc, i - 1, i)
    i = np.where((i + 1) * (2 * k - i - 2) // 2 <= pc, i + 1, i)
    j = pc - i * (2 * k - i - 1) // 2 + i + 1
    return {"main": cand[main] + 1, "pairs": np.stack([i + 1, j + 1], axis=1), "stat_main": stat[main], "stat_pairs": stat[~main]}
