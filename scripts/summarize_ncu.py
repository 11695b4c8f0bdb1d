#!/usr/bin/env python
"""Turn ncu outputs brought back in gpurun_out/ into the small text summaries kept under profiles/.
  python scripts/summarize_ncu.py launches gpurun_out/launches.csv  > profiles/<name>.txt
  python scripts/summarize_ncu.py report   gpurun_out/prof.ncu-rep  > profiles/<name>.txt
  python scripts/summarize_ncu.py traffic  gpurun_out/launches_dram.csv profiles/<name>.json > profiles/<name>.txt
      (csv from: ncu --profile-from-start off --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum,
       sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active --clock-control none --csv python scripts/profile_step.py)"""
import collections
import csv
import re
import subprocess
import sys

KEYS = ["gpu__time_duration.sum", "dram__bytes_read.sum", "dram__bytes_write.sum",
        "gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed",
        "sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "launch__registers_per_thread",
        "launch__occupancy_limit_registers", "launch__occupancy_limit_shared_mem", "launch__grid_size",
        "sm__inst_executed.avg.per_cycle_active", "sm__instruction_throughput.avg.pct_of_peak_sustained_active",
        "l1tex__throughput.avg.pct_of_peak_sustained_elapsed", "lts__throughput.avg.pct_of_peak_sustained_elapsed",
        "l1tex__data_bank_conflicts_pipe_lsu_mem_shared_op_ldgsts.sum", "smsp__inst_executed.sum",
        "l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum", "l1tex__t_requests_pipe_lsu_mem_global_op_ld.sum",
        # shared-memory data pipe: wavefronts issued for tensor-core operand fetches (UTCMMA) vs ordinary LDS / STS
        "l1tex__data_pipe_tc_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed",
        "l1tex__data_pipe_lsu_wavefronts_mem_shared.sum.pct_of_peak_sustained_elapsed",
        "l1tex__data_pipe_lsu_wavefronts_mem_shared_op_ld.sum.pct_of_peak_sustained_elapsed",
        "l1tex__data_pipe_lsu_wavefronts_mem_shared_op_st.sum.pct_of_peak_sustained_elapsed",
        "sm__pipe_tc_cycles_active.avg.pct_of_peak_sustained_elapsed",
        "sm__mem_tensor_cycles_active.avg.pct_of_peak_sustained_elapsed",
        "smsp__mem_tensor_reads_op_utcmma_matrix_c.sum.pct_of_peak_sustained_elapsed"]


def launches(path):
    lines = [l for l in open(path) if not l.startswith("==")]
    rows = []
    for r in csv.DictReader(lines):
        if r.get("Metric Name") == "gpu__time_duration.sum":
            v = float(r["Metric Value"].replace(",", ""))
            v = v / 1e3 if r["Metric Unit"] == "ns" else (v * 1e3 if r["Metric Unit"] == "ms" else v)
            rows.append((re.sub(r"\(.*", "", r["Kernel Name"]).replace("aicam::<unnamed>::", ""), r["Grid Size"], v))
    tot = sum(r[2] for r in rows)
    print("launches %d, summed kernel time %.1f us (cold-cache, serialised: compare shares)" % (len(rows), tot))
    agg = collections.defaultdict(lambda: [0, 0.0])
    for k, g, v in rows:
        agg[k][0] += 1
        agg[k][1] += v
    for k, (n, v) in sorted(agg.items(), key=lambda x: -x[1][1]):
        print("%-34s n=%3d %10.1f us %6.1f%%" % (k[:34], n, v, 100 * v / tot))
    print("\nper launch, in order:")
    for i, (k, g, v) in enumerate(rows):
        print("%3d %-28s grid %-16s %9.1f us" % (i, k[:28], g, v))


def traffic(path, json_out=None, crops=None):
    """Launch list with DRAM bytes and tensor-pipe activity per launch + the per-step totals of the tcgen05
    convolution kernels (what bench.py reports as roofline.traffic)."""
    import json
    lines = [l for l in open(path) if not l.startswith("==")]
    by_id = collections.OrderedDict()
    for r in csv.DictReader(lines):
        k = r["ID"]
        e = by_id.setdefault(k, {"name": re.search(r"(\w+_kernel)", r["Kernel Name"]).group(1) if re.search(r"(\w+_kernel)", r["Kernel Name"]) else r["Kernel Name"][:30],
                                 "full": r["Kernel Name"], "grid": r["Grid Size"]})
        v = float(r["Metric Value"].replace(",", ""))
        u = r["Metric Unit"]
        m = r["Metric Name"]
        if m == "gpu__time_duration.sum":
            e["us"] = v / 1e3 if u == "ns" else (v * 1e3 if u == "ms" else v)
        elif m.startswith("dram__bytes"):
            mult = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(u, 1)
            e["rd" if "read" in m else "wr"] = v * mult
        elif m.startswith("sm__pipe_tensor"):
            e["tensor"] = v
    rows = list(by_id.values())
    tot = sum(r.get("us", 0) for r in rows)
    print("ncu launch list of ONE step (scripts/profile_step.py); serialised launches: compare shares")
    print("metrics: gpu__time_duration.sum, dram__bytes_read.sum, dram__bytes_write.sum, sm__pipe_tensor_cycles_active.avg.pct_of_peak_sustained_active\n")
    agg = collections.defaultdict(lambda: [0, 0.0, 0.0, 0.0])
    for r in rows:
        a = agg[r["name"][:34]]
        a[0] += 1; a[1] += r.get("us", 0); a[2] += r.get("rd", 0); a[3] += r.get("wr", 0)
    print("%-36s %3s %10s %6s %12s %12s" % ("kernel", "n", "time_us", "share", "dram_rd_MB", "dram_wr_MB"))
    for k, (n, us, rd, wr) in sorted(agg.items(), key=lambda x: -x[1][1]):
        print("%-36s %3d %10.1f %5.1f%% %12.1f %12.1f" % (k, n, us, 100 * us / tot, rd / 1e6, wr / 1e6))
    print("total %.1f us\n\nper launch, in order:" % tot)
    for i, r in enumerate(rows):
        tp = re.search(r"<([^>]*)>", r["full"].replace("(int)", ""))
        print("%3d %-24s %-18s grid %-14s %8.1f us  rd %8.1f MB  wr %8.1f MB  tensor %5.1f%%" % (
            i, r["name"][:24], ("<" + tp.group(1).replace("unnamed", "").strip() + ">") if tp and "conv_win" in r["name"] else "", r["grid"], r.get("us", 0),
            r.get("rd", 0) / 1e6, r.get("wr", 0) / 1e6, r.get("tensor", 0)))
    conv = [r for r in rows if any(k in r["name"] for k in ("conv_win", "conv_pair", "stem_pool", "conv_tc"))]
    out = {"dram_read_bytes": sum(r.get("rd", 0) for r in conv), "dram_write_bytes": sum(r.get("wr", 0) for r in conv),
           "launches": len(conv), "kernel_time_us": sum(r.get("us", 0) for r in conv), "crops_in_step": crops,
           "source": "ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum over scripts/profile_step.py (64 streams), summed over "
                     "the tcgen05 convolution launches of one step"}
    out["dram_bytes"] = out["dram_read_bytes"] + out["dram_write_bytes"]
    if json_out:
        json.dump(out, open(json_out, "w"))


def report(path):
    out = subprocess.run(["ncu", "-i", path, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(out.splitlines()))
    hdr, units = rows[0], rows[1]
    for vals in rows[2:]:
        print("kernel:", vals[hdr.index("Kernel Name")][:100], "grid", vals[hdr.index("Grid Size")],
              "block", vals[hdr.index("Block Size")])
        for k in KEYS:
            if k in hdr:
                i = hdr.index(k)
                print("  %-75s %s %s" % (k, vals[i], units[i]))
    src = subprocess.run(["ncu", "-i", path, "--page", "source", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(src.splitlines()))
    if len(rows) > 2:
        hdr, data = rows[1], rows[2:]
        isrc, iex, ismp = hdr.index("Source"), hdr.index("Instructions Executed"), hdr.index("# Samples")
        tot = sum(int(r[iex]) for r in data if r[iex].isdigit())
        print("\nwarp instructions executed: %d; top SASS lines by stall samples:" % tot)
        stall = [i for i, h in enumerate(hdr) if h.startswith("stall_") and "Not Issued" not in h]
        tsm = sum(int(r[ismp]) for r in data if r[ismp].isdigit())
        for r in sorted(data, key=lambda r: -int(r[ismp]) if r[ismp].isdigit() else 0)[:14]:
            st = sorted(((int(r[i]), hdr[i]) for i in stall if r[i].isdigit()), reverse=True)[:2]
            print("  %5.1f%%  executed %9s  %-46s %s" % (100 * int(r[ismp]) / max(1, tsm), r[iex], r[isrc].strip()[:46], st))


if __name__ == "__main__":
    if sys.argv[1] == "traffic":
        traffic(sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else None, int(sys.argv[4]) if len(sys.argv) > 4 else None)
    else:
        {"launches": launches, "report": report}[sys.argv[1]](sys.argv[2])
