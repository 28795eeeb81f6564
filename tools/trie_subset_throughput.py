"""Cost of cutting a trie subset: ppd_trie_subset_[sorted_]leaves_dev against the root entry on the same leaves.

For each size, leaves are generated on the device sorted by construction (synth.gen_sorted_leaves_dev: 32-byte keys,
70-80-byte values) and permuted with torch.randperm.  Queries are random: half of them leaf keys, half random keys
(absent).  For each (order, m), after warm-up, `runs` rounds alternate the root entry and the subset entry:
  sorted     ppd_trie_root_sorted_leaves_dev / ppd_trie_subset_sorted_leaves_dev on the sorted leaves
  permuted   ppd_trie_root_leaves_dev / ppd_trie_subset_leaves_dev on the permuted leaves
gpu_ms is the library's event time of the call: every kernel, the subset stage included, not the copy of the output.
d2h_ms is a device-to-page-locked-host copy of as many bytes as the subset has, timed on its own with CUDA events.
Touched nodes are counted in the output (its branches, extensions and leaves).  The card's name and power limit are read
in the same run.

    python tools/trie_subset_throughput.py [--sizes 10000000,100000000] [--queries 1000,100000,1000000] [--runs 5]
                                           [--out profiles/r06_trie_subset.json] [--profile FILE]

--profile FILE: for each size, one sorted subset call with 100 k queries (or the largest below) under torch.profiler
(a run of its own, not timed); its per-kernel device times go to FILE.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from unsorted_leaves_throughput import gpu_info  # noqa: E402


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def count_nodes(b):
    """node kinds of a Trie in the pre-order Node form (include/ppd_flat.h)"""
    counts = [0] * 5
    p, left = 0, [1]  # nodes still to read at each open level: the Trie, then the 16 children of each open branch
    while left:
        if left[-1] == 0:
            left.pop()
            if left:  # a branch's children are done: its value follows
                p += 4 + int.from_bytes(b[p : p + 4], "little")
            continue
        left[-1] -= 1
        k = b[p]
        counts[k] += 1
        if k == 0:
            p += 1
        elif k == 1:
            p += 33
        elif k == 2:
            p += 1
            left.append(16)
        elif k == 3:
            p += 2 + b[p + 1]
            left[-1] += 1  # its child follows
        else:
            p += 2 + b[p + 1]
            p += 4 + int.from_bytes(b[p : p + 4], "little")
    assert p == len(b)
    return dict(zip(("empty", "hash", "branch", "extension", "leaf"), counts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="10000000,100000000")
    ap.add_argument("--queries", default="1000,100000,1000000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_trie_subset.json"))
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()

    import torch

    from proof_protocol_decoder_b200 import synth
    from proof_protocol_decoder_b200.lib import Context

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ctx = Context(0)
    result = {"card": gpu_info(), "runs": args.runs, "warmup": args.warmup, "sizes": {}}
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for n in [int(float(s)) for s in args.sizes.split(",")]:
        keys, off, vals = synth.gen_sorted_leaves_dev(n, seed=n % 1000 + 1)
        g = torch.Generator(device="cuda")
        g.manual_seed(n)
        pk, po, pv = synth.permute_leaves_dev(keys, off, vals, torch.randperm(n, generator=g, device="cuda"))
        torch.cuda.synchronize()
        rows = {}
        for m in [int(float(s)) for s in args.queries.split(",")]:
            pick = torch.randint(0, n, (m - m // 2,), device="cuda", generator=g)
            q = torch.cat([keys[pick], torch.randint(0, 256, (m // 2, 32), dtype=torch.uint8, device="cuda", generator=g)])
            q = q[torch.randperm(m, generator=g, device="cuda")].contiguous()
            torch.cuda.synchronize()
            calls = {
                "sorted": (lambda: ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel()),
                           lambda: ctx.trie_subset_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel(), q.data_ptr(), m)),
                "permuted": (lambda: ctx.trie_root_leaves_dev(pk.data_ptr(), 32, po.data_ptr(), pv.data_ptr(), n, pv.numel()),
                             lambda: ctx.trie_subset_leaves_dev(pk.data_ptr(), 32, po.data_ptr(), pv.data_ptr(), n, pv.numel(), q.data_ptr(), m)),
            }
            for order, (root_call, subset_call) in calls.items():
                for _ in range(args.warmup):
                    want = root_call()
                    root, sub = subset_call()
                if root != want:
                    raise SystemExit(f"n={n} m={m} {order}: the subset entry's root differs from the root entry's")
                g_root, g_sub = [], []
                for _ in range(args.runs):
                    root_call()
                    g_root.append(ctx.stats()["gpu_ms"])
                    subset_call()
                    g_sub.append(ctx.stats()["gpu_ms"])
                st = ctx.stats()
                # the output's copy on its own: as many bytes, device to page-locked host
                dev = torch.empty(len(sub), dtype=torch.uint8, device="cuda")
                host = torch.empty(len(sub), dtype=torch.uint8, pin_memory=True)
                d2h = []
                for _ in range(args.runs):
                    ev0.record()
                    host.copy_(dev, non_blocking=True)
                    ev1.record()
                    ev1.synchronize()
                    d2h.append(ev0.elapsed_time(ev1))
                del dev, host
                row = {"root_gpu_ms": summary(g_root), "subset_gpu_ms": summary(g_sub), "d2h_ms": summary(d2h), "out_bytes": len(sub),
                       "touched": count_nodes(sub) if m <= 100_000 else None, "kernel_launches": st["kernel_launches"], "root": root.hex()}
                row["added_gpu_ms"] = row["subset_gpu_ms"]["median"] - row["root_gpu_ms"]["median"]
                row["added_vs_root"] = row["added_gpu_ms"] / row["root_gpu_ms"]["median"]
                rows[f"{order}/{m}"] = row
                print(json.dumps({"n": n, "order": order, "m": m, "root_ms": round(row["root_gpu_ms"]["median"], 3),
                                  "subset_ms": round(row["subset_gpu_ms"]["median"], 3), "added": round(row["added_vs_root"], 4),
                                  "d2h_ms": round(row["d2h_ms"]["median"], 3), "out_bytes": len(sub)}), flush=True)
            if args.profile and m == max(x for x in [int(float(s)) for s in args.queries.split(",")] if x <= 100_000):
                from torch.profiler import ProfilerActivity, profile

                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    calls["sorted"][1]()
                with open(args.profile, "a") as f:
                    f.write(f"n = {n}, m = {m}: one sorted subset call\n")
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30) + "\n")
            del q
        result["sizes"][str(n)] = rows
        del keys, off, vals, pk, po, pv
        torch.cuda.empty_cache()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
