"""Every output of every solver variant on fixed inputs, one .npy file per array, so that two builds of the library can be
compared bit for bit:

    PAREBEN_LIB=libA.so python scripts/solver_outputs.py outA
    PAREBEN_LIB=libB.so python scripts/solver_outputs.py outB
    python scripts/solver_outputs.py --compare outA outB

Variants: gm (bundled Gaussian 1000 x 481, 10 folds, the 400-row grid, with and without the Gram organisation), ge
(the Epis slice of tests/golden/gauss_epis_slice.npz and the yeast matrix), bt (config 2: bundled binomial, 5 folds,
the full grid, int8 tensor-core contraction), bm (config 2's design with one entry set to 12, which keeps the FP64
contraction), be (the binomial Epis slice), and the streaming kernels (bundled Gaussian main effects, the K = 2,000
config-5 slice with Epis).  Per CV workload: fold error, status, n_selected, n_iter of run_fits and the counters
(model flops, the avoided and tensor-core entries); kernel times go to *_time.npy, which --compare skips.  Per
variant: the fit_batch records of fold 0 (all rows) on 20 grid rows."""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
REPEATS = 3          # run_fits calls per workload: the first is a warm-up, every call must give the same arrays


def golden(name):
    return np.load(os.path.join(ROOT, "tests", "golden", name))


def workloads():
    import pareben_b200 as pb
    from pareben_b200.synth import config5
    b = golden("inputs_bundled.npz")
    Xg, yg = b["BASIS"].astype(float), b["y"]
    Xb, yb = b["BASISbinomial"].astype(float), b["yBinomial"].astype(float)
    Xb12 = Xb.copy(); Xb12[7, 9] = 12.0

    def full_grid(X, y, nf, prior):
        folds = pb.AssignToFolds(X, nf)
        with pb.Problem(X, y, folds, nf, False, prior) as p:
            grid = pb.cross_validate._grid_from_lambda_max(p.lambda_max())
        idx = np.arange(grid["alpha"].size * nf)
        return folds, (idx % nf + 1, grid["alpha"][idx // nf], grid["lambda"][idx // nf])

    def slice_fits(g, nf):
        rows = g["rows"]
        idx = np.arange(rows.size * nf)
        return idx % nf + 1, g["grid_alpha"][rows][idx // nf], g["grid_lambda"][rows][idx // nf]

    fg, gm_fits = full_grid(Xg, yg, 10, "gaussian")
    fb, bt_fits = full_grid(Xb, yb, 5, "binomial")
    ges = golden("gauss_epis_slice.npz"); yeast = golden("yeast_epi008.npz"); bes = golden("binom_epis_slice.npz")
    k2 = golden("stream_k2000.npz")
    d5 = config5(int(k2["n"]), int(k2["k"]), int(k2["seed"]))
    gi, fi = np.nonzero(np.isfinite(k2["fold_err"]))
    # name: (X, y, fold_id, n_folds, epis, prior, mode, PAREBEN_GRAM, fits)
    return {
        "gm_gram1": (Xg, yg, fg, 10, False, "gaussian", pb.MODE_CACHED, "1", gm_fits),
        "gm_gram0": (Xg, yg, fg, 10, False, "gaussian", pb.MODE_CACHED, "0", gm_fits),
        "ge_slice": (Xg[:120, :25], yg[:120], ges["fold_id"], 3, True, "gaussian", pb.MODE_CACHED, None, slice_fits(ges, 3)),
        "ge_yeast": (yeast["X"].astype(float), yeast["y"], yeast["fold_id"], 10, True, "gaussian", pb.MODE_CACHED, None, slice_fits(yeast, 10)),
        "bt_config2": (Xb, yb, fb, 5, False, "binomial", pb.MODE_CACHED, None, bt_fits),
        "bm_config2_x12": (Xb12, yb, fb, 5, False, "binomial", pb.MODE_CACHED, None, bt_fits),
        "be_slice": (Xb[::4, :20], yb[::4], bes["fold_id"], 3, True, "binomial", pb.MODE_CACHED, None, slice_fits(bes, 3)),
        "stream_gm": (Xg, yg, fg, 10, False, "gaussian", pb.MODE_STREAMING, None, gm_fits),
        "stream_ge_k2000": (d5["X"].astype(float), d5["y"], k2["fold_id"], int(k2["n_folds"]), True, "gaussian", pb.MODE_STREAMING,
                            None, (fi + 1, k2["alpha"][gi], k2["lam"][gi])),
    }


def run(out_dir):
    import pareben_b200 as pb
    pb.load()
    os.makedirs(out_dir, exist_ok=True)
    save = lambda name, a: np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a))
    for name, (X, y, folds, nf, epis, prior, mode, gram, fits) in workloads().items():
        if gram is None:
            os.environ.pop("PAREBEN_GRAM", None)
        else:
            os.environ["PAREBEN_GRAM"] = gram
        pb.set_mode(mode)
        try:
            with pb.Problem(X, y, folds, nf, epis, prior) as p:
                assert p.streaming == (mode == pb.MODE_STREAMING), name
                f, a, l = (np.asarray(v) for v in fits)
                ms, first = [], None
                for _ in range(REPEATS):
                    res = p.run_fits(f.astype(np.int32), a, l)
                    flops, t, _launches = p.counters()
                    counters = np.array([flops, p.gram_info()[1], p.contraction_info()[1]])
                    if first is None:
                        first = (res, counters)
                    else:
                        assert all(u.tobytes() == v.tobytes() for u, v in zip(first[0], res)), f"{name}: repeat differs"
                        ms.append(t)
                if name.startswith("gm"):
                    assert p.gram_info()[0] == (gram == "1"), name
                if name.startswith("bm"):
                    assert p.contraction_info() == (False, 0), name
                if name.startswith("bt"):
                    assert p.contraction_info()[0], name
                for key, v in zip(("fold_err", "status", "n_selected", "n_iter"), first[0]):
                    save(f"{name}_{key}", v)
                save(f"{name}_counters", first[1])
                save(f"{name}_time", ms)
            if name not in ("gm_gram0", "ge_yeast"):     # one record set per variant: fold 0 (all rows) needs a problem without folds
                with pb.Problem(X, y, None, 0, epis, prior) as p:
                    assert p.streaming == (mode == pb.MODE_STREAMING), name
                    pick = np.unique(np.linspace(0, a.size - 1, 20).astype(int))
                    rec = p.fit_batch(np.zeros(pick.size, np.int32), np.zeros(pick.size, np.int32), a[pick], l[pick])
                for key, v in rec.items():
                    save(f"{name}_record_{key}", v)
            print(f"{name}: {f.size} fits, kernel ms {['%.2f' % t for t in ms]}", flush=True)
        finally:
            pb.set_mode(pb.MODE_AUTO)
            os.environ.pop("PAREBEN_GRAM", None)


def compare(a_dir, b_dir):
    names = sorted(n for n in os.listdir(a_dir) if n.endswith(".npy"))
    assert names == sorted(n for n in os.listdir(b_dir) if n.endswith(".npy")), "different file sets"
    bad = 0
    for n in names:
        if n.endswith("_time.npy"):
            continue
        a, b = np.load(os.path.join(a_dir, n)), np.load(os.path.join(b_dir, n))
        same = a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()
        bad += not same
        print(f"{'equal' if same else 'DIFFERENT':9s} {n} {a.shape}")
    for n in names:
        if n.endswith("_time.npy"):
            print(f"time {n[:-9]}: {np.load(os.path.join(a_dir, n))} vs {np.load(os.path.join(b_dir, n))} ms")
    print(f"{len([n for n in names if not n.endswith('_time.npy')]) - bad} equal, {bad} different")
    return bad == 0


if __name__ == "__main__":
    if len(sys.argv) == 4 and sys.argv[1] == "--compare":
        sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    run(sys.argv[1])
