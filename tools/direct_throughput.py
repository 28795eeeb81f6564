"""Throughput of direct pre-images (FlatBlock kind 2) against the same tries sent as a compact witness (kind 0).

Config-2-shaped blocks (bench.py's C2 parameters, no inline code: a direct pre-image carries no code) are sent both
ways -- the kind-2 form is the oracle's compact_to_direct of the same witness -- and decoded with
ppd_blocks_decode_stream, the two kinds in alternating runs.  Per kind: blocks/s, host CPU per block (host_busy_ms,
which for kind 2 includes re-spelling the pre-image as a witness), bytes uploaded per block, blocks that ran the device
txn loop, and the spread over the runs.  The two kinds' outputs are compared block by block first.

    python tools/direct_throughput.py [--blocks 64] [--runs 3] [--scale 1.0] [--out profiles/direct_throughput.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from concurrent.futures import ProcessPoolExecutor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True
# bench.py's C2_PARAMS (the benchmark's config-2 shape)
C2_PARAMS = dict(contract_frac=0.15, slots_lo=1, slots_hi=256, virtual_depth=7, virtual_accounts_log16=7, slot_reads=(0, 10), slot_writes=(0, 10),
                 allow_new_accounts=False, allow_self_destruct=True, inline_code_frac=0.02)


def _pair(a):
    """(kind-0 FlatBlock, kind-2 FlatBlock) of one config-2-shaped block"""
    seed, scale = a
    import ppd_oracle_lib
    from proof_protocol_decoder_b200 import flat, synth

    params = dict(C2_PARAMS, inline_code_frac=0.0)
    blk = synth.gen_block(seed, n_accounts=max(10, int(20000 * scale)), n_txns=max(2, int(200 * scale)),
                          accounts_per_txn=(80, 120) if scale >= 0.5 else (2, 8), **params)
    f0 = blk.flat
    direct = ppd_oracle_lib.load().compact_to_direct(flat.pre_image_of(f0)[1])
    return f0, flat.with_pre_image(f0, flat.PRE_IMAGE_DIRECT, direct)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "error": str(e)}


def run(ctx, flats):
    outs = [None] * len(flats)

    def done(i, r):
        if isinstance(r, Exception):
            outs[i] = r
            return
        with r:
            outs[i] = len(r.view)

    t0 = time.perf_counter()
    ctx.blocks_decode_stream(flats, done)
    dt = time.perf_counter() - t0
    bad = [o for o in outs if isinstance(o, Exception)]
    if bad:
        raise RuntimeError(f"{len(bad)} blocks failed: {bad[0]}")
    return dt, ctx.stats()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=64)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--procs", type=int, default=min(32, os.cpu_count() or 1))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from proof_protocol_decoder_b200.lib import Context

    t0 = time.perf_counter()
    with ProcessPoolExecutor(args.procs) as ex:
        pairs = list(ex.map(_pair, [(100 + i, args.scale) for i in range(args.blocks)]))
    gen_s = time.perf_counter() - t0
    kinds = {"kind0": [p[0] for p in pairs], "kind2": [p[1] for p in pairs]}
    ctx = Context(0)
    # the same tries, the same IrDump
    for i, (f0, f2) in enumerate(pairs):
        if ctx.block_decode(f0) != ctx.block_decode(f2):
            raise SystemExit(f"block {i}: kind 0 and kind 2 decode differently")
    for k in kinds:  # warm-up: every lane's buffers at their size
        run(ctx, kinds[k])
    res = {k: [] for k in kinds}
    for _ in range(args.runs):
        for k, flats in kinds.items():
            dt, st = run(ctx, flats)
            n = len(flats)
            res[k].append({"blocks_per_s": n / dt, "host_busy_ms_per_block": st["host_busy_ms"] / n, "h2d_bytes_per_block": st["h2d_bytes"] / n,
                           "txn_loops_on_gpu": st["txn_loops_on_gpu"], "witnesses_on_gpu": st["witnesses_on_gpu"]})
    ctx.close()
    summary = {}
    for k, rows in res.items():
        bps = [r["blocks_per_s"] for r in rows]
        hb = [r["host_busy_ms_per_block"] for r in rows]
        summary[k] = {"blocks_per_s_median": statistics.median(bps), "blocks_per_s_min": min(bps), "blocks_per_s_max": max(bps),
                      "host_busy_ms_per_block_median": statistics.median(hb), "host_busy_ms_per_block_min": min(hb), "host_busy_ms_per_block_max": max(hb),
                      "h2d_bytes_per_block": rows[-1]["h2d_bytes_per_block"], "txn_loops_on_gpu": rows[-1]["txn_loops_on_gpu"], "runs": rows}
    out = {"blocks": args.blocks, "scale": args.scale, "flat_bytes_per_block": {k: sum(map(len, v)) / len(v) for k, v in kinds.items()},
           "generate_s": gen_s, **gpu_info(), "result": summary}
    s = json.dumps(out, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
