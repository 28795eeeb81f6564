"""Cost of taking trie leaves in any order: ppd_trie_root_leaves_dev against ppd_trie_root_sorted_leaves_dev.

For each size, leaves are generated on the device sorted by construction (synth.gen_sorted_leaves_dev: 32-byte keys,
70-80-byte values) and permuted with torch.randperm.  Three runs per round, alternating, after warm-up:
  sorted     the sorted entry on the sorted leaves
  unsorted   the new entry on the permuted leaves (same root as `sorted`, checked)
  hashed     the new entry on the permuted leaves with PPD_LEAVES_HASH_KEYS (the 32-byte keys hashed first)
Each call ends in a device synchronise (the root is copied back); the time is the host clock around it, and gpu_ms is
the library's own event time of the call.  The card's name and power limit are read in the same run.

    python tools/unsorted_leaves_throughput.py [--sizes 1000000,10000000,100000000] [--runs 5] [--warmup 2]
                                               [--out profiles/r04_unsorted_leaves.json] [--profile FILE]

--profile FILE: after the timed runs of each size, one `unsorted` call under torch.profiler (a run of its own, not
timed); its per-kernel device times go to FILE (one table per size).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "error": str(e)}


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000,100000000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_unsorted_leaves.json"))
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()

    import torch

    from proof_protocol_decoder_b200 import synth
    from proof_protocol_decoder_b200.lib import LEAVES_HASH_KEYS, Context

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ctx = Context(0)
    result = {"card": gpu_info(), "runs": args.runs, "warmup": args.warmup, "sizes": {}}
    for n in [int(float(s)) for s in args.sizes.split(",")]:
        keys, off, vals = synth.gen_sorted_leaves_dev(n, seed=n % 1000 + 1)
        g = torch.Generator(device="cuda")
        g.manual_seed(n)
        pk, po, pv = synth.permute_leaves_dev(keys, off, vals, torch.randperm(n, generator=g, device="cuda"))
        torch.cuda.synchronize()
        calls = {
            "sorted": lambda: ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel()),
            "unsorted": lambda: ctx.trie_root_leaves_dev(pk.data_ptr(), 32, po.data_ptr(), pv.data_ptr(), n, pv.numel()),
            "hashed": lambda: ctx.trie_root_leaves_dev(pk.data_ptr(), 32, po.data_ptr(), pv.data_ptr(), n, pv.numel(), flags=LEAVES_HASH_KEYS),
        }
        roots = {}
        for _ in range(args.warmup):
            for k, f in calls.items():
                roots[k] = f()
        if roots["sorted"] != roots["unsorted"]:
            raise SystemExit(f"n={n}: the new entry's root differs from the sorted entry's")
        wall = {k: [] for k in calls}
        gpu = {k: [] for k in calls}
        for _ in range(args.runs):
            for k, f in calls.items():
                t0 = time.perf_counter()
                f()
                wall[k].append((time.perf_counter() - t0) * 1e3)
                gpu[k].append(ctx.stats()["gpu_ms"])
        row = {"value_bytes": int(vals.numel()), "root": roots["sorted"].hex(), "wall_ms": {k: summary(v) for k, v in wall.items()},
               "gpu_ms": {k: summary(v) for k, v in gpu.items()}}
        base = row["wall_ms"]["sorted"]["median"]
        row["overhead_vs_sorted"] = {k: row["wall_ms"][k]["median"] / base - 1 for k in ("unsorted", "hashed")}
        result["sizes"][str(n)] = row
        print(json.dumps({"n": n, "wall_ms": {k: round(v["median"], 2) for k, v in row["wall_ms"].items()},
                          "overhead": {k: round(v, 3) for k, v in row["overhead_vs_sorted"].items()}}), flush=True)
        if args.profile:
            from torch.profiler import ProfilerActivity, profile

            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                calls["unsorted"]()
            with open(args.profile, "a") as f:
                f.write(f"n = {n}: one unsorted call\n")
                f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30) + "\n")
        del keys, off, vals, pk, po, pv
        torch.cuda.empty_cache()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
