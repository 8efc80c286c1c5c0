"""Turn a .ncu-rep (brought back in gpurun_out/) into the text summary committed under profiles/.
usage: python tools/ncu_summary.py gpurun_out/prof.ncu-rep [top_lines] > profiles/rNN_name.txt"""
import csv, io, subprocess, sys

rep = sys.argv[1]
top = int(sys.argv[2]) if len(sys.argv) > 2 else 12
raw = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(raw)))
hdr, units = rows[0], rows[1]
WANT = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed", "dram__cycles_active.avg.pct_of_peak_sustained_elapsed",
        "sm__throughput.avg.pct_of_peak_sustained_elapsed", "l1tex__throughput.avg.pct_of_peak_sustained_active",
        "lts__throughput.avg.pct_of_peak_sustained_elapsed", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum",
        "smsp__thread_inst_executed_per_inst_executed.ratio", "launch__registers_per_thread", "launch__grid_size",
        "launch__block_size", "launch__occupancy_limit_registers", "launch__occupancy_limit_shared_mem",
        "launch__shared_mem_per_block_dynamic", "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum", "l1tex__t_requests_pipe_lsu_mem_global_op_ld.sum",
        "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum"]
idx = [hdr.index(w) for w in WANT if w in hdr]
stalls = [i for i, h in enumerate(hdr) if "smsp__average_warp" in h and "issue_stalled" in h and "ratio" in h and "not_issued" not in h]
print(f"# ncu --set full --clock-control none summary of {rep.split('/')[-1]} (per launch; cold-cache, serialised replays)")
for r in rows[2:]:
    print("\n## " + r[hdr.index("Kernel Name")])
    for i in idx:
        print(f"  {hdr[i]:<72} {r[i]:>16} {units[i]}")
    try:
        U = {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0}
        ir, iw, it = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("gpu__time_duration.sum")
        rd = float(r[ir].replace(",", "")) * U[units[ir]]
        wr = float(r[iw].replace(",", "")) * U[units[iw]]
        t = float(r[it].replace(",", "")) * {"s": 1.0, "ms": 1e-3, "us": 1e-6, "ns": 1e-9}[units[it]]
        print(f"  {'traffic = dram read + write':<72} {(rd + wr) / 1e6:>16.3f} MB  -> {(rd + wr) / t / 1e9:.1f} GB/s")
    except Exception as e:
        print("  (traffic n/a)", e)
    s = sorted(((float(r[i].replace(",", "")) if r[i] else 0, hdr[i]) for i in stalls), reverse=True)[:6]
    print("  top stalls (warp cycles per issued instr): " + ", ".join(f"{h.split('issue_stalled_')[1].split('_per')[0]}={v:.2f}" for v, h in s))
# per-source-line instruction shares of each distinct kernel
names = []
for r in rows[2:]:
    n = r[hdr.index("Kernel Name")]
    if n not in names:
        names.append(n)
for n in names:
    short = n.split("(")[0].replace("void ", "").strip()   # e.g. "stn_bwd_col_kernel<0, 2, 0>"
    src = subprocess.run(["ncu", "-i", rep, "--page", "source", "--csv", "--print-source", "cuda,sass", "--kernel-name",
                          "regex:" + short.split("<")[0].split("::")[-1], "--launch-count", "1"], capture_output=True, text=True).stdout
    agg, cur = [], None
    for r in csv.reader(io.StringIO(src)):
        if not r:
            continue
        if r[0] == "File Path":
            cur = r[1].split("/")[-1]
        elif r[0].isdigit() and len(r) > 7:
            try:
                agg.append((int(r[7].replace(",", "")), int(r[6].replace(",", "") or 0), cur, int(r[0]), r[1].strip()[:100]))
            except ValueError:
                pass
    tot = sum(a[0] for a in agg) or 1
    print(f"\n## hottest source lines (first launch matching {short.split('<')[0]}): warp instructions, share, stall samples")
    for k, smp, f, l, text in sorted(agg, reverse=True)[:top]:
        print(f"  {k:>10} {100 * k / tot:5.1f}%  smp={smp:<6} {f}:{l}  {text}")
