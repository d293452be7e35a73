"""The final models of T responses: T calls of EBelasticNet_Gaussian / _Binomial (one problem upload, one single-fit launch
and one teardown each) against one EBelasticNetMulti (one upload, one pareben_fit_batch launch), T in {1, 16, 256}.
Writes profiles/r05_final_models.md (or --out).

  gaussian   bundled Gaussian 1000 x 481 and T - 1 seeded permutations of its response
  binomial   bundled binomial 500 x 481 (genotype codes: the int8 tensor-core contraction) and T - 1 permutations

Each response is fitted at one grid point of its own BuildGrid grid, drawn with a fixed seed.  Wall time is taken
around whole calls; each call ends in a device synchronise (its results are on the host when it returns).  The two
routes alternate, after one warm-up of each; every EBelasticNetMulti result is checked key for key against the single
calls (PAREBEN_GRAM pinned to 1, so both routes take the same Gaussian organisation)."""
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


def responses(y, T, seed=2027):
    rng = np.random.default_rng(seed)
    return np.column_stack([y] + [rng.permutation(y) for _ in range(T - 1)])


def points(pb, X, Y, seed=5):
    """(lambda, alpha) per response: a seeded row of each response's own BuildGrid grid (one lambda_max pass for all)."""
    with pb.Problem(X, Y, None, 0) as p:
        lm = p.lambda_max_multi()
    rows = np.random.default_rng(seed).integers(0, 400, Y.shape[1])
    gs = [pb.cross_validate._grid_from_lambda_max(float(v)) for v in lm]
    return np.array([g["lambda"][r] for g, r in zip(gs, rows)]), np.array([g["alpha"][r] for g, r in zip(gs, rows)])


def same(a, b):
    if set(a) != set(b):
        return False
    return all(np.array_equal(a[k], b[k]) if isinstance(a[k], np.ndarray) else a[k] == b[k] for k in a)


def run(pb, name, X, y, prior, Ts, reps):
    single = pb.EBelasticNet_Gaussian if prior == "gaussian" else pb.EBelasticNet_Binomial
    lines = []
    for T in Ts:
        Y = responses(y, T)
        L, A = points(pb, X, Y)
        pb.EBelasticNetMulti(X, Y[:, :1], L[:1], A[:1], prior=prior)          # warm: modules, pools
        single(X, Y[:, 0], L[0], A[0])
        tm, ts = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            multi = pb.EBelasticNetMulti(X, Y, L, A, prior=prior)
            tm.append(time.perf_counter() - t0)
            t0 = time.perf_counter()
            singles = [single(X, Y[:, t], L[t], A[t]) for t in range(T)]
            ts.append(time.perf_counter() - t0)
            assert all(same(m, s) for m, s in zip(multi, singles)), f"{name} T={T}: EBelasticNetMulti differs from the single calls"
        n_eff = np.array([m["weight"].shape[0] for m in multi])
        m_ms, s_ms = 1e3 * min(tm), 1e3 * min(ts)
        lines.append(f"| {name} | {T} | {n_eff.min()} / {int(np.median(n_eff))} / {n_eff.max()} | {s_ms:.1f} | {m_ms:.1f} | "
                     f"{s_ms / m_ms:.2f}x | {s_ms / T:.2f} | {m_ms / T:.3f} |")
        print(lines[-1], flush=True)
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_final_models.md"))
    ap.add_argument("--T", type=int, nargs="+", default=[1, 16, 256])
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    os.environ["PAREBEN_GRAM"] = "1"
    import pareben_b200 as pb
    if pb.device_count() < 1:
        raise SystemExit("needs a CUDA device")
    g = np.load(os.path.join(ROOT, "tests", "golden", "inputs_bundled.npz"))
    which = card()
    lines = run(pb, "Gaussian 1000x481", g["BASIS"], g["y"], "gaussian", a.T, a.reps)
    lines += run(pb, "binomial 500x481", g["BASISbinomial"], g["yBinomial"], "binomial", a.T, a.reps)
    head = [
        "# Final models of T responses: T EBelasticNet calls against one EBelasticNetMulti", "",
        f"Card: {which} (name, power limit, read in the same run).  `python scripts/final_models.py`; best of {a.reps} alternating "
        "runs after one warm-up of each route.  Responses: the bundled response and T - 1 seeded permutations, each at a seeded "
        "point of its own BuildGrid grid; PAREBEN_GRAM=1.  Every EBelasticNetMulti result was equal, key for key, to the T single calls.",
        "", "Wall time around whole calls (upload, fit, read-back, teardown); each call ends in a device synchronise.", "",
        "| workload | T | weight rows min / median / max | T x EBelasticNet ms | EBelasticNetMulti ms | speed-up | ms per response, singles | ms per response, multi |",
        "|---|---|---|---|---|---|---|---|",
    ]
    with open(a.out, "w") as fh:
        fh.write("\n".join(head + lines) + "\n")
    print(f"wrote {a.out}")


if __name__ == "__main__":
    main()
