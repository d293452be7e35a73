#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the EBEN cross-validation hot path.

Workload (BASELINE.json configs[1]): CrossValidate, prior="binomial", on the reference's bundled
BASISbinomial / yBinomial (500 x 481, tests/golden/inputs_bundled.npz), nFolds = 5, Epis = "no",
the full 20 x 20 (alpha, lambda) grid  ->  2,000 independent EBEN fits per step.
One "step" = one pass of the hot path over that grid: every fit from initialisation to its
hold-out log-likelihood.

  value   whole-job fits/s with the problem already resident in HBM (pareben_run_fits), timed
          with CUDA events on the library's launch stream, max over ranks.
  e2e     the same metric through the host-buffer C-ABI call a user's CrossValidate makes
          (pareben_cv_grid): H2D of BASIS/y/folds/grid from pinned host memory, per-fold layout
          kernels, the fit kernel, D2H of the error table -- all inside the timed region.
  N > 1   one process per GPU (torchrun); STRONG scaling: the ONE 2,000-fit grid is split N ways
          (pareben_shard_plan: cost-interleaved round-robin), each rank computes its shard and the
          shards are merged by one NCCL all-reduce of the three small tables (inside the e2e region;
          the resident `value` has no collective in it because the data path has none).
  extras  the same measurement on the bundled Gaussian data (1000 x 481, 10 folds, 4,000 fits --
          four of the five BASELINE configs are Gaussian), sharded the same way; and BASELINE config 5's shape
          (synthetic n = 1,000, Epis = "yes", 10 folds, the full 4,000-fit grid) through the streaming kernels:
          k = 20,000 loci (200,010,000 candidates) when 8 GPUs share the grid, a k = 5,000 slice (12.5 M candidates)
          on fewer, with the score-contraction kernel's own time, flops and fraction of the FP64 tensor peak.
  --impl reference   times the reference's own C (oracle/_ref, compiled unmodified from
          /root/reference/EBEN_orig/src) -- or the oracle's C restatement when that library is
          absent -- on all host cores: the whole 2,000-fit grid when --steps <= 2, else a
          stratified sample of it (every lambda rank, every alpha) per step.
  --dump-outputs DIR   writes the per-fit tables the last timed step of `value` computed (hold-out error, status,
          active-set size, iterations) and its grid as DIR/<name>.npy, so that two builds can be compared output by output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
os.environ.setdefault("OPENBLAS_NUM_THREADS", "1")

import numpy as np  # noqa: E402

METRIC = "EBEN CV grid fits/sec"
UNIT = "fits/s"
WORKLOAD = "config2: CrossValidate binomial, bundled BASISbinomial 500x481 / yBinomial, nFolds=5, Epis=no, 20x20 grid = 2000 fits/step"
CONFIG = {"workload": WORKLOAD, "fits_per_step": 2000, "l2_flush_between_steps": True,
          "multi_gpu": "one grid split over the ranks (strong scaling), merged by one all-reduce"}
DATA = "bundled BASISbinomial/yBinomial (reference fixture, tests/golden/inputs_bundled.npz)"


def load_workload(which: str = "binomial"):
    g = np.load(os.path.join(ROOT, "tests", "golden", "inputs_bundled.npz"))
    if which == "binomial":
        return g["BASISbinomial"].astype(np.float64), g["yBinomial"].astype(np.float64), 5
    return g["BASIS"].astype(np.float64), g["y"].astype(np.float64), 10


def dump_outputs(out_dir: str, res, n_folds: int) -> None:
    """--dump-outputs: what pareben_run_fits returned in the last timed step, merged over the ranks, as float64 .npy files:
    per-fit tables of shape (grid row, fold) in BuildGrid's row order, and the grid they were computed on (its lambdas
    come from the device's lambda_max).  The inputs are fixed (bundled data, seeded folds), so two builds compare file by file."""
    os.makedirs(out_dir, exist_ok=True)
    grid = res["grid"]
    tables = {"fold_error": res["table"], "status": res["status"], "n_selected": res["nsel"], "iterations": res["iters"]}
    for name, a in tables.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, dtype=np.float64).reshape(grid["alpha"].size, n_folds))
    for name in ("alpha", "lambda"):
        np.save(os.path.join(out_dir, "grid_" + name + ".npy"), np.asarray(grid[name], dtype=np.float64))


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference implementation on the host cores
def _cpu_task(args):
    from oracle import rlayer as R
    X, y, fid, f, lam, a, kind = args
    e, fit = R.fit_one(X, y, fid, f, lam, a, False, "binomial", R.fit_lib(kind))
    return e


def sample_rows(n_offsets: int):
    """Grid rows of a stratified sample: for every lambda rank l (0..19) the alpha indices (7 l + 3 j) mod 20, j < n_offsets.
    Every lambda rank is visited n_offsets times and (7 is coprime to 20) every alpha value as well."""
    return sorted({20 * l + (7 * l + 3 * j) % 20 for j in range(min(n_offsets, 20)) for l in range(20)})


def cpu_run(X, y, n_folds, grid_alpha, grid_lambda, folds, rows, procs: int, pool):
    """Time the given grid rows (all folds) on `procs` worker processes, one fit per task, longest first."""
    from oracle import rlayer as R
    kind = R.available_kind()
    jobs = [(X, y, folds, f, grid_lambda[r], grid_alpha[r], kind) for r in rows for f in range(1, n_folds + 1)]
    jobs.sort(key=lambda j: j[4])                                  # small lambda = long fits first: no straggler at the end
    t0 = time.perf_counter()
    pool.map(_cpu_task, jobs, chunksize=1)
    dt = time.perf_counter() - t0
    return len(jobs), dt, kind


def cpu_pool(procs: int):
    """Worker pool for the CPU arm.  The reference library is loaded in THIS process before the fork, so that it is
    part of the parent's address space (and of what the driver's loaded-library hook sees), and inherited by the workers."""
    from multiprocessing import get_context
    from oracle import rlayer as R
    R.fit_lib(R.available_kind())
    return get_context("fork").Pool(procs)


def cpu_warm(pool, X, y, folds, ga, gl, procs):
    """Untimed: one cheap fit per worker (page-in, first-touch allocations)."""
    from oracle import rlayer as R
    pool.map(_cpu_task, [(X, y, folds, 1, gl[0], ga[0], R.available_kind())] * procs, chunksize=1)


def oracle_grid(X, y, n_folds):
    from oracle import rlayer as R
    ga, gl = R.build_grid(X, y, n_folds)
    return ga, gl, R.assign_to_folds(X.shape[0], n_folds)


def cpu_describe(rows, n_folds, n_grid, dt, procs):
    if len(rows) == n_grid:
        return f"the full grid: {n_grid} rows x {n_folds} folds = {n_grid * n_folds} fits, {dt:.1f} s wall on {procs} processes"
    lam_ranks = len({r // 20 for r in rows}); alphas = len({r % 20 for r in rows})
    return (f"stratified sample: {len(rows)} grid rows ({lam_ranks} of 20 lambda ranks, {alphas} of 20 alpha values) x {n_folds} folds = "
            f"{len(rows) * n_folds} of {n_grid * n_folds} fits, {dt:.1f} s wall on {procs} processes")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    X, y, n_folds = load_workload()
    ga, gl, folds = oracle_grid(X, y, n_folds)
    procs = os.cpu_count() or 1
    full = args.steps <= 2
    n_off = max(3, -(-10 * procs // (20 * n_folds)))              # >= 10 jobs per core
    rows = list(range(ga.size)) if full else sample_rows(n_off)
    total_fits, total_t, kind = 0, 0.0, "port"
    with cpu_pool(procs) as pool:
        cpu_warm(pool, X, y, folds, ga, gl, procs)
        for _ in range(min(args.warmup, 1)):
            cpu_run(X, y, n_folds, ga, gl, folds, sample_rows(1), procs, pool)
        for _ in range(args.steps):
            n, dt, kind = cpu_run(X, y, n_folds, ga, gl, folds, rows, procs, pool)
            total_fits += n; total_t += dt
    value = total_fits / total_t
    sample = cpu_describe(rows, n_folds, ga.size, total_t / args.steps, procs)
    line = {"metric": METRIC, "value": value, "unit": UNIT, "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps,
            "higher_is_better": True, "scaling": "strong" if args.gpus > 1 else "weak",
            "vs_baseline": None, "dtype": "f64", "data": DATA, "config": CONFIG,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "reference" if kind == "reference" else "port",
                             "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def run_gpu(args):
    import torch
    import torch.distributed as dist
    import pareben_b200 as pb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly one JSON line: anything libraries print while the run is in progress (NCCL writes its
    # version banner to stdout when the communicator comes up) is sent to stderr instead
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    pb.load()
    if pb.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (the hot path has no CPU implementation; use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    # FP64 peak for the roofline denominator (MEASURED_PEAKS.json has HBM and bf16 only)
    peak_dfma = pb.measure_fp64_peak(local, 0)
    peak_dmma = pb.measure_fp64_peak(local, 1)
    peak = max(peak_dfma, peak_dmma)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device="cuda")       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], device="cuda", dtype=torch.float64)
        dist.all_reduce(t)
        return float(t.item())

    def resident(X, y, n_folds, prior, steps, warmup, sampler=None):
        """One grid, split over the ranks, problem resident: returns per-step device ms (max over ranks), the merged table
        and this launch's algorithmic flops summed over ranks."""
        folds = pb.AssignToFolds(X, n_folds)
        prob = pb.Problem(X, y, folds, n_folds, False, prior, device=local)
        grid = pb.cross_validate._grid_from_lambda_max(prob.lambda_max())
        n_grid = grid["alpha"].size
        mine = pb.shard_plan(grid["lambda"], n_folds, rank, world)
        f_vec = (mine % n_folds + 1).astype(np.int32); a_vec = grid["alpha"][mine // n_folds]; l_vec = grid["lambda"][mine // n_folds]
        if sampler:
            sampler.start()                    # nvidia-smi needs a moment to deliver its first sample: started before the warm-up,
        for _ in range(warmup):                # read after the timed steps (same kernel, same load throughout)
            prob.run_fits(f_vec, a_vec, l_vec)
        barrier()
        ms_steps, fl_steps, av_steps, wall0 = [], [], [], time.perf_counter()
        for _ in range(steps):
            flush.zero_()                      # L2 flush between timed iterations
            torch.cuda.synchronize()
            err, st, ns, it = prob.run_fits(f_vec, a_vec, l_vec)
            fl, ms, _launches = prob.counters()
            ms_steps.append(ms); fl_steps.append(fl); av_steps.append(prob.gram_info()[1])
        barrier()
        wall = time.perf_counter() - wall0
        clocks = sampler.stop() if sampler else None
        total_ms = max_over_ranks(float(np.sum(ms_steps)))             # ranks run side by side: the job takes the slowest rank's time
        flops = sum_over_ranks(float(np.mean(fl_steps)))
        avoided = sum_over_ranks(float(np.mean(av_steps)))
        gram = prob.gram_info()[0]
        table = np.zeros(n_grid * n_folds); table[mine] = err
        stat = np.zeros(n_grid * n_folds); stat[mine] = st
        nsel = np.zeros(n_grid * n_folds); nsel[mine] = ns
        iters = np.zeros(n_grid * n_folds); iters[mine] = it
        if world > 1:
            t = torch.from_numpy(np.stack([table, stat, nsel, iters])).cuda()
            dist.all_reduce(t)
            table, stat, nsel, iters = t.cpu().numpy()
        prob.close()
        return {"ms_per_step": total_ms / steps, "flops": flops, "table": table, "status": stat, "nsel": nsel, "iters": iters, "grid": grid, "folds": folds,
                "n_fits": n_grid * n_folds, "wall": wall, "clocks": clocks, "avoided": avoided, "gram": gram, "my_ms": float(np.mean(ms_steps)), "my_fits": int(mine.size)}

    X, y, n_folds = load_workload()
    n, k = X.shape
    res = resident(X, y, n_folds, "binomial", args.steps, args.warmup, ClockSampler(local))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, n_folds)
    n_fits = res["n_fits"]
    grid, folds = res["grid"], res["folds"]
    n_grid = grid["alpha"].size
    value = n_fits / (res["ms_per_step"] * 1e-3)

    # ---- e2e: host buffers (pinned) -> pareben_cv_grid (this rank's shard) -> merged host table, every step ----
    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.from_numpy(np.empty(0, a.dtype)).dtype, pin_memory=True)
        out = t.numpy()
        out[...] = a
        return out, t
    Xp, _k1 = pinned(np.asfortranarray(X).T.copy())      # column-major bytes of X, held as a C-contiguous (k, n) array
    yp, _k2 = pinned(y); fp, _k3 = pinned(folds.astype(np.int32))
    Xcol = Xp.T                                          # (n, k) Fortran-ordered view onto the pinned block
    ap, _k4 = pinned(grid["alpha"]); lp, _k5 = pinned(grid["lambda"])

    def e2e_step():
        e, s, m = pb.cv_grid(Xcol, yp, fp, n_folds, ap, lp, prior="binomial", device=local, shard=rank, n_shards=world)
        return pb.cross_validate._merge_shards(e, s, m, local)          # the `.combine = rbind` of the reference: one all-reduce

    for _ in range(min(args.warmup, 2)):
        e2e_step()                       # also brings the NCCL communicator up outside the timed region
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        e_err, e_st, e_ns = e2e_step()
    barrier()
    e2e_t = max_over_ranks(time.perf_counter() - t0)
    e2e_value = n_fits * args.steps / e2e_t
    my_fits = res["my_fits"]
    h2d = X.nbytes + y.nbytes + folds.size * 4 + 2 * n_grid * 8 + my_fits * 40            # per rank: data + grid + task list
    d2h = my_fits * (8 + 12) + 8
    assert np.array_equal(e_err.ravel(), res["table"]), "e2e and resident paths disagree"

    # ---- extras: the bundled Gaussian grid, sharded the same way (fewer steps: it is the longer grid) ----
    extras = {}
    if not args.no_extras:
        Xg, yg, nfg = load_workload("gaussian")
        g_steps = max(1, min(args.steps, 3))
        rg = resident(Xg, yg, nfg, "gaussian", g_steps, 1)
        g_ach = rg["flops"] / (rg["ms_per_step"] * 1e-3) / 1e12
        extras["gaussian_bundled_1000x481_10fold"] = {
            "fits_per_step": rg["n_fits"], "ms_per_step": rg["ms_per_step"], "fits_per_s": rg["n_fits"] / (rg["ms_per_step"] * 1e-3),
            "steps": g_steps, "algorithmic_tflops": g_ach, "roofline_frac": g_ach / (peak * world),
            # the Gram organisation shares the candidate cache between the fits of a fold: the model's contraction flops for it are not executed
            "gram_organisation": bool(rg["gram"]), "executed_tflops": (rg["flops"] - rg["avoided"]) / (rg["ms_per_step"] * 1e-3) / 1e12,
            "status_nonzero": int((rg["status"] != 0).sum()), "max_active_set": int(rg["nsel"].max())}

        if not args.no_stream:
            from pareben_b200.synth import config5
            ks = args.stream_k if args.stream_k > 0 else (20000 if world >= 8 else 5000)
            d5 = config5(1000, ks)
            X5 = d5["X"].astype(np.float64); y5 = d5["y"]
            folds5 = pb.AssignToFolds(X5, 10)
            t_lm = time.perf_counter()
            grid5 = pb.BuildGrid(X5, y5, 10, "yes", device=local)
            t_lm = time.perf_counter() - t_lm
            mine5 = pb.shard_plan(grid5["lambda"], 10, rank, world)
            pb.set_mode(pb.MODE_STREAMING)
            try:
                with pb.Problem(X5, y5, folds5, 10, True, "gaussian", device=local) as p5:
                    barrier()
                    t5 = time.perf_counter()
                    e5, st5, ns5, it5 = p5.run_fits((mine5 % 10 + 1).astype(np.int32), grid5["alpha"][mine5 // 10], grid5["lambda"][mine5 // 10])
                    _fl5, ms5, launches5 = p5.counters()
                    scan_ms, scan_fl, scans, rounds = p5.stream_counters()
                    barrier()
                    wall5 = max_over_ranks(time.perf_counter() - t5)
            finally:
                pb.set_mode(pb.MODE_AUTO)
            job_ms = max_over_ranks(ms5)
            tot_scan_fl = sum_over_ranks(scan_fl); max_scan_ms = max_over_ranks(scan_ms)
            extras["config5_streaming"] = {
                "workload": f"synthetic n=1000 x k={ks} Gaussian, Epis=yes ({ks * (ks + 1) // 2} candidates), 10 folds, 20x20 grid = 4000 fits, one grid split over the ranks",
                "fits_per_step": 4000, "ms_per_step": job_ms, "fits_per_s": 4000 / (job_ms * 1e-3), "wall_s": wall5, "steps": 1,
                "lambda_max_s": t_lm, "rounds": rounds, "kernel_launches_rank0": launches5,
                "scan_kernel": {"name": "stream_scan_kernel<epis>", "launches_rank0": scans, "ms_total_max_over_ranks": max_scan_ms,
                                "algorithmic_tflop": tot_scan_fl / 1e12, "achieved_tflops": tot_scan_fl / (max_scan_ms * 1e-3) / 1e12,
                                "roofline_frac": tot_scan_fl / (max_scan_ms * 1e-3) / 1e12 / (peak_dmma * world)},
                "status_nonzero": int(sum_over_ranks(float((st5 != 0).sum()))), "max_active_set": int(max_over_ranks(float(ns5.max())))}

    if rank == 0:
        achieved = res["flops"] / (res["ms_per_step"] * 1e-3) / 1e12
        cpu = None
        if world == 1 and not args.no_cpu:
            ga, gl, ofolds = oracle_grid(X, y, n_folds)
            procs = os.cpu_count() or 1
            rows = sample_rows(max(3, -(-10 * procs // (20 * n_folds))))
            with cpu_pool(procs) as pool:
                cpu_warm(pool, X, y, ofolds, ga, gl, procs)
                nj, dt, kind = cpu_run(X, y, n_folds, ga, gl, ofolds, rows, procs, pool)
            cpu = {"value": nj / dt, "unit": UNIT, "cores": procs, "kind": "reference" if kind == "reference" else "port",
                   "sample": cpu_describe(rows, n_folds, ga.size, dt, procs)}
        traffic = None
        for name in ("r02_traffic.json", "r01_traffic.json"):
            tp = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tp):
                try:
                    traffic = json.load(open(tp)).get("dram_bytes_per_launch")
                    break
                except Exception:
                    traffic = None
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "strong" if world > 1 else "weak",
                "vs_baseline": None, "dtype": "f64", "data": DATA, "config": CONFIG,
                "extras": dict(extras, status_nonzero=int((res["status"] != 0).sum()), max_active_set=int(res["nsel"].max()),
                               fits_on_rank0=my_fits, rank0_kernel_ms=res["my_ms"]),
                "clocks": res["clocks"],
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d * world), "d2h_bytes_per_step": int(d2h * world),
                        "ms_per_step": 1e3 * e2e_t / args.steps},
                "gpu_launches": int(args.steps * world),
                "roofline": {"bound": "tensor", "pipe": "fp64 (DMMA mma.sync.m8n8k4.f64 for the contraction, DFMA elsewhere)",
                             "achieved": achieved, "peak": peak * world, "unit": "TFLOP/s", "frac": achieved / (peak * world),
                             "traffic": traffic, "kernel": "eben_fit_kernel<binomial,main>",
                             "algorithmic_flops_per_launch": res["flops"], "launch_ms": res["ms_per_step"],
                             "peak_source": f"on-box probe at bench start: DFMA {peak_dfma:.1f}, DMMA {peak_dmma:.1f} TFLOP/s per GPU "
                                            "(MEASURED_PEAKS.json has no FP64 entry)"},
                "cpu_baseline": cpu, "wall_s_timed_region": res["wall"]}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps of the headline measurement and of e2e (the Gaussian extra runs min(steps, 3), "
                         "the streaming extra one)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the Gaussian extras")
    ap.add_argument("--no-stream", action="store_true", help="skip the config-5 streaming extra")
    ap.add_argument("--stream-k", type=int, default=0, help="loci of the config-5 streaming extra (0: 20000 on 8 GPUs, else 5000)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the tables the last timed step of the headline measurement computed as DIR/<name>.npy "
                         "(float64), as soon as that measurement ends; add --no-cpu --no-extras for a quick comparison run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
