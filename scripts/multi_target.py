"""One multi-response call against T single-response calls, T in {1, 4, 16}, on four workloads; writes
profiles/r04_multi_target.md (or --out).  Responses are the workload's own response and T - 1 seeded permutations of
it (what a permutation threshold runs); each gets its own BuildGrid grid.  Multi and single runs alternate.

  config2     binomial bundled 500 x 481, 5 folds, full 20 x 20 grid (the bench.py workload)
  gaussian    bundled Gaussian 1000 x 481, 10 folds, full grid
  lambda_max  GetLambdaMax of an Epis design, config-5 recipe, n = 1000, K = 5,000 (12.5 M pairs)
  streaming   the same K = 5,000 design, Epis, 10 folds, streaming mode, 10 x 10 sub-grid per response

Per workload and T: "resident" = the fit call on problems already uploaded (pareben_problem_cv_grid[_multi]); "e2e" =
upload + lambda_max + fits + teardown (what CrossValidateMulti / T CrossValidate calls pay), wall clock.
Every multi table is checked against the single tables with np.array_equal (PAREBEN_GRAM pinned to 1)."""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:          # noqa: BLE001
        return f"unknown ({e})"


def responses(y, T, seed=2026):
    rng = np.random.default_rng(seed)
    return np.column_stack([y] + [rng.permutation(y) for _ in range(T - 1)])


def grids(pb, X, Y, epis, rows):
    with pb.Problem(X, Y, None, 0, epis) as p:
        lm = p.lambda_max_multi()
    gs = [pb.cross_validate._grid_from_lambda_max(float(v)) for v in lm]
    return np.stack([g["alpha"][rows] for g in gs]), np.stack([g["lambda"][rows] for g in gs])


def sync_time(fn):
    t = time.perf_counter()
    out = fn()
    return time.perf_counter() - t, out


def fit_workload(pb, name, X, y, n_folds, epis, prior, rows, Ts, reps, stream=False):
    folds = pb.AssignToFolds(X, n_folds)
    lines = []
    for T in Ts:
        Y = responses(y, T)
        A, L = grids(pb, X, Y, epis, rows)
        n_fits = A.size * n_folds
        if stream:
            pb.set_mode(pb.MODE_STREAMING)
        try:
            res_m, res_s, e2e_m, e2e_s = [], [], [], []
            with pb.Problem(X, Y, folds, n_folds, epis, prior) as p:
                singles = [pb.Problem(X, Y[:, t], folds, n_folds, epis, prior) for t in range(T)]
                p.cv_grid_multi(A[:, :1], L[:, :1])                     # warm: modules, Gram matrices, pools
                for t in range(T):
                    singles[t].cv_grid(A[t, :1], L[t, :1])
                for _ in range(reps):
                    dt, tm = sync_time(lambda: p.cv_grid_multi(A, L))
                    res_m.append(dt)
                    dt, ts = sync_time(lambda: [singles[t].cv_grid(A[t], L[t]) for t in range(T)])
                    res_s.append(dt)
                    for i in range(3):
                        assert np.array_equal(tm[i], np.stack([s[i] for s in ts])), f"{name} T={T}: tables differ"
                for s in singles:
                    s.close()
            for _ in range(reps if not stream else 0):
                def multi_e2e():
                    with pb.Problem(X, Y, folds, n_folds, epis, prior) as q:
                        lm = q.lambda_max_multi()
                        q.cv_grid_multi(A, L)
                    return lm

                def single_e2e():
                    for t in range(T):
                        with pb.Problem(X, Y[:, t], folds, n_folds, epis, prior) as q:
                            q.lambda_max()
                            q.cv_grid(A[t], L[t])
                e2e_m.append(sync_time(multi_e2e)[0])
                e2e_s.append(sync_time(single_e2e)[0])
        finally:
            pb.set_mode(pb.MODE_AUTO)
        rm, rs = min(res_m), min(res_s)
        e2e = f"{min(e2e_m) * 1e3:.1f} / {min(e2e_s) * 1e3:.1f} ms ({min(e2e_s) / min(e2e_m):.2f}x)" if e2e_m else "not measured"
        lines.append(f"| {name} | {T} | {n_fits} | {rm * 1e3:.1f} | {rs * 1e3:.1f} | {rs / rm:.2f}x | {n_fits / rm:,.0f} | "
                     f"{n_fits / rs:,.0f} | {e2e} |")
        print(lines[-1], flush=True)
    return lines


def lambda_max_workload(pb, X, y, Ts, reps):
    lines = []
    for T in Ts:
        Y = responses(y, T)
        with pb.Problem(X, Y, None, 0, True) as p:
            singles = [pb.Problem(X, Y[:, t], None, 0, True) for t in range(T)]
            p.lambda_max_multi()
            singles[0].lambda_max()
            tm, ts = [], []
            for _ in range(reps):
                dt, lm = sync_time(p.lambda_max_multi)
                tm.append(dt)
                dt, ls = sync_time(lambda: [s.lambda_max() for s in singles])
                ts.append(dt)
                assert np.array_equal(lm, np.array(ls)), "lambda_max differs"
            for s in singles:
                s.close()
        m, s = min(tm), min(ts)
        lines.append(f"| lambda_max Epis K=5000 | {T} | - | {m * 1e3:.1f} | {s * 1e3:.1f} | {s / m:.2f}x | - | - | - |")
        print(lines[-1], flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_multi_target.md"))
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--T", type=int, nargs="+", default=[1, 4, 16])
    ap.add_argument("--skip-stream", action="store_true")
    a = ap.parse_args()
    import pareben_b200 as pb
    from pareben_b200.synth import config5
    pb.load()
    if pb.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    os.environ["PAREBEN_GRAM"] = "1"
    g = np.load(os.path.join(ROOT, "tests", "golden", "inputs_bundled.npz"))
    full = np.arange(400)
    sub = (np.arange(0, 20, 2)[:, None] * 20 + np.arange(0, 20, 2)[None, :]).ravel()
    head = ["| workload | T | fits | multi resident ms | T singles resident ms | speed-up | multi fits/s | singles fits/s | "
            "e2e multi / singles |", "|---|---|---|---|---|---|---|---|---|"]
    lines = []
    lines += fit_workload(pb, "config2 binomial 500x481, 5 folds, 400 points", g["BASISbinomial"].astype(np.float64), g["yBinomial"],
                          5, False, "binomial", full, a.T, a.reps)
    lines += fit_workload(pb, "Gaussian 1000x481, 10 folds, 400 points", g["BASIS"].astype(np.float64), g["y"], 10, False, "gaussian",
                          full, a.T, a.reps)
    d5 = config5(1000, 5000)
    X5 = d5["X"].astype(np.float64)
    lines += lambda_max_workload(pb, X5, d5["y"], a.T, max(a.reps, 3))
    if not a.skip_stream:
        lines += fit_workload(pb, "streaming Epis K=5000, 10 folds, 100 points", X5, d5["y"], 10, True, "gaussian", sub, a.T, 1,
                              stream=True)
    text = "\n".join([
        "# One multi-response call against T single-response calls",
        "",
        f"Card: {card()} (name, power limit).  `python scripts/multi_target.py`; best of {a.reps} alternating runs (streaming: 1, "
        "lambda_max: best of 3).  Responses: the workload's response and T - 1 seeded permutations, each with its own "
        "BuildGrid grid; PAREBEN_GRAM=1.  Every multi table was np.array_equal to the T single tables.",
        "",
        "Resident: the fit call on problems already on the device.  e2e: upload + lambda_max + fits + teardown, wall clock.",
        "",
        *head, *lines, ""])
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    open(a.out, "w").write(text)
    print(text)


if __name__ == "__main__":
    main()
