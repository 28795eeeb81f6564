"""Cost of a resident trie handle: subsets and updates of a trie kept in HBM, against rebuilding it.

For each size, leaves are generated on the device sorted by construction (synth.gen_sorted_leaves_dev: 32-byte keys,
70-80-byte values) and a handle is created from them (ppd_trie_create_sorted_leaves_dev).  Then, after warm-up, `runs`
rounds of each:
  root          ppd_trie_root_sorted_leaves_dev on the same leaves (the one-shot rebuild), alternated with
  subset/m      ppd_trie_subset_dev on the handle with m queries (half leaf keys, half random keys)
  update/k      ppd_trie_update_dev with a batch of k updates in random order: 60 % overwrites of present keys, 30 % new
                keys, 10 % deletes of present keys; 75-byte values.  Each round updates the handle further.
  update/n10    one batch of k = n / 10 (no target; no extra row when n / 10 is one of the batch sizes)
Each update grows the trie by about 20 % of k; when a buffer of the handle's spare state or leaf set outgrows its
capacity, DevBuf::reserve frees and allocates it inside the call, and that time is part of the call's gpu_ms.
gpu_ms is the library's event time of the call (sort, merge, structure and hashing for an update; not the output's copy
for a subset); nodes_hashed is what the update re-hashed.  handle_bytes is the drop of cudaMemGetInfo's free memory over
the create.  The card's name and power limit are read in the same run.

    python tools/trie_update_throughput.py [--sizes 1000000,10000000,100000000] [--batches 1000,10000,100000]
                                           [--queries 1000,100000] [--runs 5] [--out profiles/r07_trie_update.json]
                                           [--profile FILE]

--profile FILE: for the largest size, one update of the largest batch and one subset of the largest query set under
torch.profiler (a run of its own, not timed); its per-kernel device times go to FILE.
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

VLEN = 75


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def make_batch(torch, keys, k, g):
    """k device updates: 60 % overwrites, 30 % new keys, 10 % deletes, shuffled"""
    n = keys.shape[0]
    n_ow, n_del = int(0.6 * k), int(0.1 * k)
    n_new = k - n_ow - n_del
    ow = keys[torch.randint(0, n, (n_ow,), device="cuda", generator=g)]
    de = keys[torch.randint(0, n, (n_del,), device="cuda", generator=g)]
    new = torch.randint(0, 256, (n_new, 32), dtype=torch.uint8, device="cuda", generator=g)
    uk = torch.cat([ow, new, de])
    ud = torch.cat([torch.zeros(n_ow + n_new, dtype=torch.uint8, device="cuda"), torch.ones(n_del, dtype=torch.uint8, device="cuda")])
    perm = torch.randperm(k, generator=g, device="cuda")
    uk, ud = uk[perm].contiguous(), ud[perm].contiguous()
    uo = torch.arange(k + 1, dtype=torch.int64, device="cuda") * VLEN
    uv = torch.randint(0, 256, (k * VLEN,), dtype=torch.uint8, device="cuda", generator=g)
    return uk, ud, uo, uv


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1000000,10000000,100000000")
    ap.add_argument("--batches", default="1000,10000,100000")
    ap.add_argument("--queries", default="1000,100000")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_trie_update.json"))
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()

    import torch

    from proof_protocol_decoder_b200 import synth
    from proof_protocol_decoder_b200.lib import Context

    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ctx = Context(0)
    result = {"card": gpu_info(), "runs": args.runs, "warmup": args.warmup, "value_bytes": VLEN, "sizes": {}}
    sizes = [int(float(s)) for s in args.sizes.split(",")]
    batches = [int(float(s)) for s in args.batches.split(",")]
    queries = [int(float(s)) for s in args.queries.split(",")]
    for n in sizes:
        keys, off, vals = synth.gen_sorted_leaves_dev(n, seed=n % 1000 + 1)
        g = torch.Generator(device="cuda")
        g.manual_seed(n)
        torch.cuda.synchronize()
        root_call = lambda: ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel())  # noqa: E731
        want = root_call()
        free0 = torch.cuda.mem_get_info()[0]
        t = ctx.trie_from_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel())
        create_ms = ctx.stats()["gpu_ms"]
        handle_bytes = free0 - torch.cuda.mem_get_info()[0]
        if t.root != want:
            raise SystemExit(f"n={n}: the handle's root differs from the root entry's")
        rows = {"create_gpu_ms": create_ms, "handle_bytes": handle_bytes}
        g_root = []
        for m in queries:
            pick = torch.randint(0, n, (m - m // 2,), device="cuda", generator=g)
            q = torch.cat([keys[pick], torch.randint(0, 256, (m // 2, 32), dtype=torch.uint8, device="cuda", generator=g)]).contiguous()
            torch.cuda.synchronize()
            for _ in range(args.warmup):
                t.subset_dev(q.data_ptr(), m)
            g_sub = []
            for _ in range(args.runs):
                root_call()
                g_root.append(ctx.stats()["gpu_ms"])
                sub = t.subset_dev(q.data_ptr(), m)
                g_sub.append(ctx.stats()["gpu_ms"])
            rows[f"subset/{m}"] = {"gpu_ms": summary(g_sub), "out_bytes": len(sub)}
            print(json.dumps({"n": n, "subset_m": m, "gpu_ms": round(statistics.median(g_sub), 3)}), flush=True)
            if args.profile and n == sizes[-1] and m == queries[-1]:
                from torch.profiler import ProfilerActivity, profile

                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    t.subset_dev(q.data_ptr(), m)
                with open(args.profile, "a") as f:
                    f.write(f"n = {n}: one handle subset, m = {m}\n")
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30) + "\n")
        # n / 10 gets a row of its own unless it is one of the batch sizes already
        for k in batches + ([n // 10] if n // 10 not in batches else []):
            label = f"update/{k}" if k in batches else "update/n10"
            reps = args.runs if k in batches else 1
            g_upd, hashed = [], []
            for r in range(args.warmup + reps):
                uk, ud, uo, uv = make_batch(torch, keys, k, g)
                torch.cuda.synchronize()
                t.update_dev(uk.data_ptr(), ud.data_ptr(), uo.data_ptr(), uv.data_ptr(), k, uv.numel())
                st = ctx.stats()
                if r >= args.warmup:
                    g_upd.append(st["gpu_ms"])
                    hashed.append(st["nodes_hashed"])
                    root_call()
                    g_root.append(ctx.stats()["gpu_ms"])
            rows[label] = {"k": k, "gpu_ms": summary(g_upd), "nodes_hashed": hashed, "n_after": t.n}
            print(json.dumps({"n": n, "update_k": k, "gpu_ms": round(statistics.median(g_upd), 3), "nodes_hashed": hashed[0]}), flush=True)
            if args.profile and n == sizes[-1] and k == batches[-1]:
                from torch.profiler import ProfilerActivity, profile

                uk, ud, uo, uv = make_batch(torch, keys, k, g)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    t.update_dev(uk.data_ptr(), ud.data_ptr(), uo.data_ptr(), uv.data_ptr(), k, uv.numel())
                with open(args.profile, "a") as f:
                    f.write(f"n = {n}: one handle update, k = {k}\n")
                    f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=40) + "\n")
        rows["root_gpu_ms"] = summary(g_root)
        print(json.dumps({"n": n, "root_gpu_ms": round(statistics.median(g_root), 3), "create_gpu_ms": round(create_ms, 3),
                          "handle_gb": round(handle_bytes / 1e9, 2)}), flush=True)
        result["sizes"][str(n)] = rows
        t.close()
        del keys, off, vals
        torch.cuda.empty_cache()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result["card"]))


if __name__ == "__main__":
    main()
