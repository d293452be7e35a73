"""Turn the raw captures a GPU run left in gpurun_out/ into the tracked summaries under profiles/.
usage: python scripts/make_profiles.py r01     (reads launches.csv, prof_binom_full.ncu-rep, bench*.json, parity.md)"""
import collections, csv, json, os, re, subprocess, sys

tag = sys.argv[1] if len(sys.argv) > 1 else "r01"
# optional: python scripts/make_profiles.py r01 <report.ncu-rep> <suffix> "<workload text>"  -> only profiles/<tag>_fit_kernel_<suffix>_ncu.md
ALT = sys.argv[2:5] if len(sys.argv) >= 5 else None
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROUND = f"Round {int(tag[1:])}" if tag[1:].isdigit() else tag
G = os.path.join(ROOT, "gpurun_out"); P = os.path.join(ROOT, "profiles")
os.makedirs(P, exist_ok=True)

# ---- launch list ------------------------------------------------------------------------------
if not ALT:
    rows = [r for r in csv.reader(open(os.path.join(G, "launches.csv"))) if len(r) > 10]
    hdr = rows[0]; ik, iv = hdr.index("Kernel Name"), hdr.index("Metric Value")
    agg = collections.defaultdict(lambda: [0, 0.0])
    for r in rows[1:]:
        name = re.sub(r"\(.*", "", r[ik]).replace("<unnamed>::", "").replace("pareben::", "")
        agg[name][0] += 1; agg[name][1] += float(r[iv]) / 1e6
    tot = sum(v[1] for v in agg.values())
    with open(os.path.join(P, f"{tag}_launches.md"), "w") as f:
        f.write(f"# {ROUND} -- ncu launch list of `python bench.py --steps 2 --warmup 1 --no-cpu`\n\n"
                "`ncu --metrics gpu__time_duration.sum --clock-control none -c 400 --csv` (raw: `" + f"{tag}_launches_bench_steps2.csv`). "
                "Per-launch times are cold-cache and serialised: compare shares.\n\n| kernel | launches | total ms | share |\n|---|---|---|---|\n")
        for k, (n, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"| `{k}` | {n} | {ms:.3f} | {100 * ms / tot:.2f} % |\n")
        f.write("\nThe fit kernel is the only kernel of a step (`gpu_launches` = 1 per step); `dfma_peak_kernel`/`dmma_peak_kernel` are the FP64 peak "
                "probes bench.py runs once before the timed region; the gather/transpose/scale/int8 kernels belong to `pareben_problem_create` "
                "(e2e path and set-up).\n")
    with open(os.path.join(P, f"{tag}_launches_bench_steps2.csv"), "w") as f:
        w = csv.writer(f); w.writerow(["id", "kernel", "grid", "block", "gpu__time_duration_ns"])
        for r in rows[1:]:
            w.writerow([r[0], re.sub(r"\(.*", "", r[ik]), r[hdr.index("Grid Size")], r[hdr.index("Block Size")], r[iv]])

# ---- full capture -----------------------------------------------------------------------------
rep = ALT[0] if ALT else os.path.join(G, "prof_binom_full.ncu-rep")
raw = list(csv.reader(subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout.splitlines()))
h, u, v = raw[0], raw[1], raw[2]
want = ["gpu__time_duration.sum", "launch__grid_size", "launch__block_size", "launch__registers_per_thread", "launch__occupancy_limit_registers",
        "launch__occupancy_limit_shared_mem", "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__pipe_tensor_subpipe_dmma_cycles_active.avg.pct_of_peak_sustained_active", "sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active", "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__t_sector_hit_rate.pct", "lts__t_sector_hit_rate.pct", "dram__bytes_read.sum",
        "dram__bytes_write.sum", "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
        "l1tex__throughput.avg.pct_of_peak_sustained_elapsed", "sm__cycles_active.avg", "sm__cycles_elapsed.avg",
        "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio", "smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio",
        "smsp__average_warps_issue_stalled_wait_per_issue_active.ratio", "smsp__average_warps_issue_stalled_short_scoreboard_per_issue_active.ratio",
        "smsp__average_warps_issue_stalled_math_pipe_throttle_per_issue_active.ratio",
        "sm__pipe_tensor_cycles_active_realtime.avg.pct_of_peak_sustained_elapsed", "l1tex__t_requests_pipe_lsu_mem_local_op_ld.sum",
        "l1tex__t_requests_pipe_lsu_mem_local_op_st.sum"]
h = [x.split(".TriageCompute.")[-1] if ".TriageCompute." in x else x for x in h]
val = {k: (v[h.index(k)], u[h.index(k)]) for k in want if k in h}
def num(k):
    x, un = val[k]; x = float(x.replace(",", ""))
    return x * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}.get(un, 1.0)
dr, dw = num("dram__bytes_read.sum"), num("dram__bytes_write.sum")
if not ALT: json.dump({"kernel": "eben_fit_kernel<EPIS=0,BINOMIAL=1>", "workload": "config 2 full grid, 2000 fits, one launch (scripts/profile_case.py binomial 2000)",
           "dram_bytes_read": dr, "dram_bytes_write": dw, "dram_bytes_per_launch": dr + dw, "ncu_duration_ms": float(val["gpu__time_duration.sum"][0]),
           "source": f"ncu --set full --clock-control none, gpurun_out/prof_binom_full.ncu-rep ({tag})"}, open(os.path.join(P, f"{tag}_traffic.json"), "w"), indent=1)

# stall samples by source region (enclosing top-level function) and by line
def func_starts(path):
    out = []
    for i, ln in enumerate(open(path), 1):
        m = re.match(r"^(?:__device__|static __device__)\s+(?:inline\s+)?[\w:<> \*&]+?\s+(\w+)\s*\(", ln)
        if m: out.append((i, m.group(1)))
    return out
starts = {f: func_starts(os.path.join(ROOT, "pareben_b200", "csrc", f)) for f in ("gauss_fit.cuh", "binom_fit.cuh", "contract.cuh", "linalg.cuh", "eben_step.cuh", "common.cuh", "fit_kernel.cuh", "stream_scan.cuh", "stream_fit.cuh", "stream.cuh")}
def region(f, line):
    best = f"{f}:(top)"
    for ln, nm in starts.get(f, []):
        if ln - 3 <= line: best = nm           # template<> line(s) precede the signature
        else: break
    return best
src = list(csv.reader(subprocess.run(["ncu", "-i", rep, "--page", "source", "--print-source", "cuda,sass", "--csv"], capture_output=True, text=True).stdout.splitlines()))
cur = None; hd = None; reg = collections.defaultdict(collections.Counter); lines = []; total = 0; spills = 0; nexec = 0
for r in src:
    if not r: continue
    if r[0] == "File Path": cur = r[1].split("/")[-1]; hd = None; continue
    if r[0] == "Function Name": continue
    if r[0] == "Line No": hd = r; continue
    if hd is None: continue
    if r[2] != "-":
        try: n = int(r[hd.index("Instructions Executed")])
        except ValueError: continue
        nexec += n
        if "LDL" in r[3] or "STL" in r[3]: spills += n
        continue
    try: n = int(r[hd.index("# Samples")]); ln = int(r[0])
    except ValueError: continue
    if n <= 0: continue
    name = region(cur, ln); reg[name]["samples"] += n; total += n
    st = collections.Counter()
    for i, c in enumerate(hd):
        if c.startswith("stall_") and "Not Issued" not in c and r[i].isdigit(): reg[name][c[6:]] += int(r[i]); st[c[6:]] += int(r[i])
    lines.append((n, cur, ln, r[1].strip()[:100], st.most_common(3)))
alg = None
try:
    for ln in open(os.path.join(G, "plain_profile_full.log")): alg = ln.strip()
except OSError: pass
out_md = os.path.join(P, f"{tag}_fit_kernel_{ALT[1]}_ncu.md" if ALT else f"{tag}_fit_kernel_ncu.md")
with open(out_md, "w") as f:
    if ALT:
        f.write(f"# {ROUND} -- ncu `--set full`: {ALT[2]}\n\n| metric | value | unit |\n|---|---|---|\n")
        alg = None
    else:
        f.write(f"# {ROUND} -- ncu `--set full` of the fit kernel on the bench workload\n\n"
            "Command (on the B200 box, after the same command exited 0 without ncu): `ncu --set full --clock-control none --import-source on "
            "-k regex:eben_fit -s 1 -c 1 python scripts/profile_case.py binomial 2000`  \n"
            "Workload: config 2, all 2,000 fits, ONE launch of `eben_fit_kernel<EPIS=0,BINOMIAL=1>` (hybrid kernel: DMMA contraction fed by a cp.async ring, "
            "SIMT quadratic forms and pipelined Gram matrix for M <= 64).\n\n| metric | value | unit |\n|---|---|---|\n")
    for k in want:
        if k in val: f.write(f"| `{k}` | {val[k][0]} | {val[k][1]} |\n")
    f.write(f"\nDRAM traffic per launch = {(dr + dw) / 1e6:.1f} MB (read {dr / 1e6:.1f} + write {dw / 1e6:.1f}).  "
            f"Local-memory (register spill) instructions: {spills} of {nexec} executed ({100 * spills / max(nexec, 1):.2f} %).\n")
    if alg: f.write(f"Same command without ncu (CUDA events): `{alg}`\n")
    f.write("\n## Warp-stall samples by device function\n\n```\n" + f"total samples {total}\n")
    for name, c in sorted(reg.items(), key=lambda kv: -kv[1]["samples"])[:24]:
        st = [(k, n) for k, n in c.most_common(5) if k != "samples"][:4]
        f.write(f"{100 * c['samples'] / total:5.1f}%  {name:28s} {st}\n")
    f.write("```\n\n## Warp-stall samples by source line (top 25)\n\n```\n")
    for n, fl, ln, text, st in sorted(lines, reverse=True)[:25]:
        f.write(f"{100 * n / total:5.1f}% {fl}:{ln:>4} {text}   {st}\n")
    f.write("```\n")

# ---- bench lines and parity table ---------------------------------------------------------------
if ALT: print(open(out_md).read()[:3000]); sys.exit(0)
for a, b in (("bench.json", f"{tag}_bench_n1.json"), ("bench_reference.json", f"{tag}_bench_reference_n1.json"), ("parity.md", f"{tag}_parity.md")):
    if os.path.exists(os.path.join(G, a)): open(os.path.join(P, b), "w").write(open(os.path.join(G, a)).read())
print(open(out_md).read()[:6000])
