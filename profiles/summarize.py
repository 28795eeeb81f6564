#!/usr/bin/env python3
"""Turn the ncu captures of profiles/capture.sh (gpurun_out/<tag>_*) into the tracked summaries under
profiles/:  python profiles/summarize.py r01"""
import collections
import csv
import json
import os
import subprocess
import sys

TAG = sys.argv[1] if len(sys.argv) > 1 else "r01"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("SRC", os.path.join(ROOT, "gpurun_out"))
DST = os.environ.get("DST", os.path.join(ROOT, "profiles"))
PARSE_KERNELS = ("tile_exit", "group_exit", "top_chain", "tile_entry", "tile_mark", "ins_scatter", "ins_info", "heights_kernel", "min64_i16",
                 "link_kernel16", "shape_kernel", "scan_block_kernel", "scan_add_kernel", "emit_kernel", "climb_kernel", "code_list", "totals_kernel")


def launches(path):
    rows = [r for r in csv.reader(open(path, errors="replace")) if len(r) > 10]
    hdr = rows[0]
    L = collections.OrderedDict()
    for r in rows[1:]:
        d = dict(zip(hdr, r))
        e = L.setdefault(d["ID"], {"kernel": d["Kernel Name"].split("(")[0].replace("void ", "").replace("ppd::", ""), "grid": d["Grid Size"], "stream": d["Stream"]})
        try:
            e[d["Metric Name"]] = float(d["Metric Value"].replace(",", ""))
        except ValueError:
            pass
    return list(L.values())


def kernel_table(items, title):
    agg = collections.OrderedDict()
    for o in items:
        a = agg.setdefault(o["kernel"], [0, 0.0, 0.0])
        a[0] += 1
        a[1] += o.get("gpu__time_duration.sum", 0.0)
        a[2] += o.get("dram__bytes_read.sum", 0.0) + o.get("dram__bytes_write.sum", 0.0)
    tot = sum(a[1] for a in agg.values()) or 1.0
    out = [title, f"{'kernel':60s} {'launches':>8s} {'time us':>12s} {'share':>7s} {'dram MB':>10s}"]
    for k, a in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        out.append(f"{k[:60]:60s} {a[0]:8d} {a[1] / 1e3:12.1f} {100 * a[1] / tot:6.1f}% {a[2] / 1e6:10.1f}")
    return "\n".join(out)


def raw_page(rep, metrics):
    txt = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(txt.splitlines()))
    hdr = rows[0]
    idx = {h: i for i, h in enumerate(hdr)}
    out = []
    for r in rows[2:]:
        out.append({m: r[idx[m]] for m in ["Kernel Name", "Grid Size"] + metrics if m in idx})
    return out


FULL = ["gpu__time_duration.sum", "sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active", "smsp__issue_active.avg.pct_of_peak_sustained_active",
        "sm__warps_active.avg.pct_of_peak_sustained_active", "smsp__inst_executed.sum", "smsp__thread_inst_executed_per_inst_executed.ratio",
        "launch__registers_per_thread", "dram__bytes_read.sum", "dram__bytes_write.sum", "l1tex__data_bank_conflicts_pipe_lsu_mem_shared.sum",
        "smsp__average_warps_issue_stalled_math_pipe_throttle_per_issue_active.ratio", "smsp__average_warps_issue_stalled_long_scoreboard_per_issue_active.ratio"]
SHORT = ["time", "alu_pipe%", "issue%", "warps%", "warp_inst", "thr/inst", "regs", "dram_rd", "dram_wr", "smem_conflicts", "stall_math_throttle", "stall_long_sb"]


def full_table(rep, title):
    rows = raw_page(rep, FULL)
    out = [title, "kernel | grid | " + " | ".join(SHORT)]
    for r in rows:
        out.append(f"{r['Kernel Name'].split('(')[0].replace('void ', '')[:34]:34s} | {r['Grid Size']:14s} | " + " | ".join(str(r.get(m, ''))[:11] for m in FULL))
    return "\n".join(out), rows


def main():
    # ---- config 2 launch list ----
    p = os.path.join(SRC, f"{TAG}_launches_c2.csv")
    if os.path.exists(p):
        items = launches(p)
        open(os.path.join(DST, f"{TAG}_launches_c2_summary.txt"), "w").write(
            "ncu launch list of the bench command (profiles/capture*.sh says which: r01 64 blocks per step, first 4000 launches; r02 4 blocks per step, all launches; --metrics gpu__time_duration.sum,dram__bytes_*;\n"
            "--clock-control none).  Launches are serialised and cold-cache under ncu: read SHARES, not absolutes.\n\n"
            + kernel_table(items, f"all {len(items)} launches") + "\n\n"
            + kernel_table([o for o in items if "at::" not in o["kernel"] and "native" not in o["kernel"]], "this library's kernels only") + "\n")
        for o in items:
            o["kernel"] = o["kernel"].replace("<unnamed>::", "").replace("unnamed>::", "")
        ours = [o for o in items if o["kernel"].startswith(("hash_level", "keccak256_batch"))]
        hl = [o for o in ours if o["kernel"].startswith("hash_level")]
        traffic = sum(o.get("dram__bytes_read.sum", 0) + o.get("dram__bytes_write.sum", 0) for o in hl) / max(1, len(hl))
        json.dump({"kernel": "hash_level_kernel", "launches_in_capture": len(hl), "dram_bytes_per_launch_mean": traffic,
                   "time_ns_per_launch_mean_under_ncu": sum(o.get("gpu__time_duration.sum", 0) for o in hl) / max(1, len(hl)),
                   "source": f"gpurun_out/{TAG}_launches_c2.csv (ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum, all hash_level_kernel launches of the bench command)"},
                  open(os.path.join(DST, f"{TAG}_traffic.json"), "w"), indent=1)
    # ---- full capture of the level kernel (one block) ----
    rep = os.path.join(SRC, f"{TAG}_hash_level_full.ncu-rep")
    if os.path.exists(rep):
        t, _ = full_table(rep, "ncu --set full, hash_level_kernel, the level launches of one device-resident replay of one C2 block\n(PPD_HOST_THREADS=1, --blocks-per-step 1; launch-skip / launch-count as in profiles/capture*.sh)")
        open(os.path.join(DST, f"{TAG}_hash_level_full.txt"), "w").write(t + "\n")
    rep = os.path.join(SRC, f"{TAG}_txn_loop_full.ncu-rep")
    if os.path.exists(rep):
        more = ["smsp__average_warps_issue_stalled_barrier_per_issue_active.ratio", "smsp__average_warps_issue_stalled_short_scoreboard_per_issue_active.ratio",
                "smsp__warps_active.avg.per_cycle_active", "l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum"]
        rows = raw_page(rep, FULL + more)
        out = ["ncu --set full, txn_loop_kernel: two launches (16 txns each) of one config-2 block's loop (one thread block of 256 threads)", ""]
        for r in rows:
            out.append(r["Kernel Name"].split("(")[0] + "  grid " + r["Grid Size"])
            for m in FULL + more:
                if m in r:
                    out.append(f"  {m:95s} {r[m]}")
        open(os.path.join(DST, f"{TAG}_txn_loop_full.txt"), "w").write("\n".join(out) + "\n")
    rep = os.path.join(SRC, f"{TAG}_dump_full.ncu-rep")
    if os.path.exists(rep):
        t, _ = full_table(rep, "ncu --set full, ir_size_kernel + ir_emit_kernel of one config-2 block (200 IRs, one thread block of 1 024 threads each; the third decode of `profiles/run_parse.py 3`)")
        open(os.path.join(DST, f"{TAG}_dump_full.txt"), "w").write(t + "\n")
    # ---- config 5 ----
    p = os.path.join(SRC, f"{TAG}_launches_c5.csv")
    if os.path.exists(p):
        items = [o for o in launches(p) if "at::" not in o["kernel"] and "native" not in o["kernel"] and "at_cuda" not in o["kernel"]]
        txt = "ncu launch list of `python profiles/run_c5.py 10000000 1` (sorted leaves resident in HBM -> root), this library's kernels:\n\n" + kernel_table(items, "")
        txt += "\n\nper launch:\n" + "\n".join(f"{o['kernel'][:40]:40s} {o['grid']:16s} {o.get('gpu__time_duration.sum', 0) / 1e3:10.1f} us  dram {(o.get('dram__bytes_read.sum', 0) + o.get('dram__bytes_write.sum', 0)) / 1e6:9.1f} MB" for o in items)
        open(os.path.join(DST, f"{TAG}_launches_c5_summary.txt"), "w").write(txt + "\n")
    rep = os.path.join(SRC, f"{TAG}_c5_full.ncu-rep")
    if os.path.exists(rep):
        t, _ = full_table(rep, "ncu --set full, the hashing kernels of config 5 at 10M leaves (first 14 hash_* launches)")
        open(os.path.join(DST, f"{TAG}_c5_full.txt"), "w").write(t + "\n")
    # ---- witness parse / arena kernels ----
    p = os.path.join(SRC, f"{TAG}_launches_parse.csv")
    if os.path.exists(p):
        items = [o for o in launches(p) if "at::" not in o["kernel"] and "native" not in o["kernel"] and "at_cuda" not in o["kernel"]]
        for o in items:
            o["kernel"] = o["kernel"].replace("<unnamed>::", "").replace("unnamed>::", "")
        last = max(i for i, o in enumerate(items) if o["kernel"].startswith("tile_exit"))
        one = items[last:]
        txt = ("ncu launch list of `python profiles/run_parse.py 2` (one config-2 block, 34.6 MB witness, 1.05 M instructions, one lane):\n"
               "the kernels of the LAST decode, in launch order.  Serialised and cold-cache under ncu: read SHARES; the plain run's\n"
               "CUDA-event time of the parse phases is in " + f"{TAG}_parse_plain.log.\n\n")
        agg = collections.OrderedDict()
        for o in one:
            a = agg.setdefault(o["kernel"], [0, 0.0, 0.0, 0.0])
            a[0] += 1
            a[1] += o.get("gpu__time_duration.sum", 0.0)
            a[2] += o.get("dram__bytes_read.sum", 0.0)
            a[3] += o.get("dram__bytes_write.sum", 0.0)
        tot = sum(a[1] for a in agg.values()) or 1.0
        txt += f"{'kernel':44s} {'launches':>8s} {'time us':>10s} {'share':>7s} {'dram rd MB':>11s} {'dram wr MB':>11s}\n"
        for k, a in agg.items():
            txt += f"{k[:44]:44s} {a[0]:8d} {a[1] / 1e3:10.1f} {100 * a[1] / tot:6.1f}% {a[2] / 1e6:11.1f} {a[3] / 1e6:11.1f}\n"
        txt += f"{'total':44s} {'':8s} {tot / 1e3:10.1f}\n"
        open(os.path.join(DST, f"{TAG}_launches_parse_summary.txt"), "w").write(txt)
    rep = os.path.join(SRC, f"{TAG}_parse_full.ncu-rep")
    if os.path.exists(rep):
        t, rows = full_table(rep, "ncu --set full, the witness parse / arena kernels of one config-2 block (both decodes of `profiles/run_parse.py 2`; the second one is warm)")
        open(os.path.join(DST, f"{TAG}_parse_full.txt"), "w").write(t + "\n")
    for f in (f"{TAG}_bench_plain.log", f"{TAG}_c5_plain.log", f"{TAG}_parse_plain.log"):
        if os.path.exists(os.path.join(SRC, f)):
            open(os.path.join(DST, f), "w").write(open(os.path.join(SRC, f)).read())


def count_parse_kernels(path):
    """number of ppd_parse.cu launches in one decode (the last one of the launch list)"""
    items = launches(path)
    for o in items:
        o["kernel"] = o["kernel"].replace("<unnamed>::", "").replace("unnamed>::", "")
    last = max(i for i, o in enumerate(items) if o["kernel"].startswith("tile_exit"))
    return sum(1 for o in items[last:] if o["kernel"].startswith(PARSE_KERNELS))


def count_kernel(path, name, blocks):
    """launches of kernel `name` per block decode: the launches before the first replay (3 warm-up decodes of `blocks`
    blocks each would need the program's structure; simpler: the level launches between two consecutive tile_exit launches)"""
    items = launches(path)
    for o in items:
        o["kernel"] = o["kernel"].replace("<unnamed>::", "").replace("unnamed>::", "")
    # the last decode of the capture runs one lane at a time only when blocks == 1; count over the whole capture instead
    firsts = [i for i, o in enumerate(items) if o["kernel"].startswith("tile_exit")]
    n_decodes = len(firsts)
    # decodes are followed by replays (no tile_exit in a HASH replay): count the launches up to the first replay, i.e.
    # within the first blocks * 3 decodes there are blocks * 3 * per_block of them
    upto = firsts[min(len(firsts) - 1, blocks * 3)] if n_decodes > blocks * 3 else len(items)
    n = sum(1 for o in items[:upto] if o["kernel"].startswith(name))
    return n // (blocks * 3)


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--count-parse-kernels":
        print(count_parse_kernels(sys.argv[2]))
    elif len(sys.argv) > 4 and sys.argv[1] == "--count-kernel":
        print(count_kernel(sys.argv[2], sys.argv[3], int(sys.argv[4])))
    else:
        main()
