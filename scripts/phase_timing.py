"""Experiments only: per-phase cycle totals of the fit kernel (needs libpareben_timing.so, built with
-DPAREBEN_PHASE_TIMING).  usage: PAREBEN_LIB=pareben_b200/libpareben_timing.so python scripts/phase_timing.py [binomial|gaussian]"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import pareben_b200 as pb
lib = pb.load()
lib.pareben_phase_cycles.restype = ctypes.c_int
lib.pareben_phase_cycles.argtypes = [ctypes.POINTER(ctypes.c_ulonglong), ctypes.c_int]
names = ["vfill", "contract", "quad", "gram", "sweep", "irls(all, incl. gram+sweep)", "delta_ml", "actions", "loglik/resid", "refresh(other)",
         "  irls: predictor + line search", "  irls: weights, direction, tests", "  irls: H -> SIGMA copy", "  sweep: loads + stores"]
g = np.load("tests/golden/inputs_bundled.npz")
prior = sys.argv[1] if len(sys.argv) > 1 else "binomial"
if prior == "binomial":
    X, y, nf = g["BASISbinomial"].astype(float), g["yBinomial"].astype(float), 5
else:
    X, y, nf = g["BASIS"].astype(float), g["y"], 10
folds = pb.AssignToFolds(X, nf); grid = pb.BuildGrid(X, y, nf)
fold = np.tile(np.arange(1, nf + 1), 400); a = np.repeat(grid["alpha"], nf); l = np.repeat(grid["lambda"], nf)
if prior != "binomial":
    sel = np.arange(0, fold.size, 4); fold, a, l = fold[sel], a[sel], l[sel]
with pb.Problem(X, y, folds, nf, False, prior) as p:
    p.run_fits(fold, a, l)
    buf = (ctypes.c_ulonglong * 32)()
    lib.pareben_phase_cycles(buf, 1)
    p.run_fits(fold, a, l)
    fl, ms, _ = p.counters()
    n = lib.pareben_phase_cycles(buf, 1)
    cyc = np.array(buf[:n], dtype=float); calls = np.array(buf[n:2 * n], dtype=float)
    total_block_cycles = ms * 1e-3 * 1.965e9 * 296
    print(f"{prior}: kernel {ms:.1f} ms, {fold.size} fits; block-cycles available ~ {total_block_cycles:.3e}")
    lib.pareben_fit_trace.restype = ctypes.c_int
    nf_ = fold.size
    t0 = np.zeros(nf_, np.uint64); t1 = np.zeros(nf_, np.uint64); blk = np.zeros(nf_, np.int32)
    which = 0 if prior != 'binomial' else (4 if p.contraction_info()[0] else 2)      # bt: the tensor-core variant
    got = lib.pareben_fit_trace(which, t0.ctypes.data_as(ctypes.c_void_p), t1.ctypes.data_as(ctypes.c_void_p), blk.ctypes.data_as(ctypes.c_void_p), nf_)
    if got:
        start = t0.min(); dur = (t1 - t0).astype(float) * 1e-6; end = (t1.max() - start) * 1e-6
        busy = dur.sum() / (end * (blk.max() + 1))
        order = np.argsort(-dur)
        print(f"  fit trace: span {end:.1f} ms, blocks {blk.max()+1}, busy fraction {busy:.3f}; fit ms: max {dur.max():.1f} p99 {np.quantile(dur,0.99):.1f} median {np.median(dur):.2f} mean {dur.mean():.2f}")
        print("  longest fits (ms, lambda, alpha, start ms):", [(round(dur[i],1), float(l[i]), float(a[i]), round(float(t0[i]-start)*1e-6,1)) for i in order[:5]])
        lastend = np.array([ (t1[blk==b].max()-start)*1e-6 for b in range(blk.max()+1)])
        print(f"  block finish times ms: min {lastend.min():.1f} median {np.median(lastend):.1f} max {lastend.max():.1f}")
        err, st, ns, it = p.run_fits(fold, a, l)
        os.makedirs("gpurun_out", exist_ok=True)
        np.savez_compressed(f"gpurun_out/trace_{prior}.npz", dur_ms=dur, start_ms=(t0 - start).astype(float) * 1e-6, block=blk, lam=l, alpha=a, fold=fold, n_sel=ns, n_iter=it)
    for nm, c, k in zip(names, cyc, calls):
        print(f"  {nm:30s} {c:.3e}  {100*c/total_block_cycles:5.1f} % of block time   calls {k:.0f}  cycles/call {c/max(k,1):.0f}")
