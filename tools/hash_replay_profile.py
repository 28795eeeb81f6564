#!/usr/bin/env python3
"""Where the hashing replay's time goes: the C2 replay that bench.py reports as device_ms_per_step.hashing, timed, then
one torch.profiler pass of it.

  python tools/hash_replay_profile.py --out DIR [--steps 20] [--blocks 64]

Builds the lanes bench.py builds (64 C2 blocks, seeds 2..65, every block decoded 8 times in one stream call, so each
lane keeps the last block it decoded resident), then:
  * replay_last(REPLAY_HASH) --steps times, the L2 overwritten (256 MiB) before every step as bench.py does; the mean
    and every step's time go to DIR/replay.json;
  * one more step under torch.profiler with CUDA activities: per-kernel totals (DIR/kernels.txt), each lane's
    (stream's) launches (DIR/timeline.json), and in DIR/summary.json the tail (the first lane's last kernel end to the
    last lane's last kernel end) and the share of the step spent in level launches of at most 4 CTAs (512 nodes).
The card's name, power limit and SM clock limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import bench  # noqa: E402  (sets CUDA_DEVICE_MAX_CONNECTIONS before torch creates the context)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:200]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--blocks", type=int, default=64)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)

    seeds = [2 + j for j in range(args.blocks)]
    flats = bench.c2_blocks(seeds, 1.0, os.cpu_count() or 1)
    os.environ.setdefault("PPD_HOST_THREADS", str(args.blocks))

    import torch
    from torch.profiler import ProfilerActivity, profile

    from proof_protocol_decoder_b200.lib import Context

    torch.cuda.set_device(0)
    ctx = Context(0)
    flats = [ctx.pinned_copy(f) for f in flats]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def decode(mult):
        done = []

        def on_done(i, o):
            if isinstance(o, Exception):
                raise o
            done.append(o.nbytes)
            o.close()

        ctx.blocks_decode_stream(flats * mult, on_done)
        assert len(done) == len(flats) * mult

    for _ in range(3):
        decode(8)
    lanes = ctx.replay_lanes()

    def step():
        flush.zero_()
        torch.cuda.synchronize()
        return ctx.replay_last(ctx.REPLAY_HASH)

    for _ in range(3):
        step()
    ms = [step() for _ in range(args.steps)]
    info = {"card": card(), "lanes": lanes, "steps": args.steps, "l2": "256 MiB written before every step",
            "ms_mean": sum(ms) / len(ms), "ms_min": min(ms), "ms_max": max(ms), "ms": ms}
    json.dump(info, open(os.path.join(args.out, "replay.json"), "w"), indent=1)
    print(f"hashing replay: {info['ms_mean']:.3f} ms/step (min {min(ms):.3f}, max {max(ms):.3f}) over {lanes} lanes", flush=True)

    # ---- one profiled step ----
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
    with open(os.path.join(args.out, "kernels.txt"), "w") as f:
        f.write(prof.key_averages().table(sort_by="cuda_time_total", row_limit=30))
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "trace.json")
        prof.export_chrome_trace(path)
        trace = json.load(open(path))
    kern = [e for e in trace.get("traceEvents", []) if e.get("cat") == "kernel" and "flush" not in e.get("name", "").lower()
            and "fill" not in e.get("name", "").lower() and "elementwise" not in e.get("name", "").lower()]
    by_stream = {}
    for e in kern:
        a = e.get("args", {})
        by_stream.setdefault(str(a.get("stream", e.get("tid"))), []).append(
            {"name": e["name"][:80], "ts_us": e["ts"], "dur_us": e["dur"], "grid": a.get("grid"), "block": a.get("block")})
    t0 = min(e["ts"] for e in kern)
    t1 = max(e["ts"] + e["dur"] for e in kern)
    for s in by_stream.values():
        s.sort(key=lambda k: k["ts_us"])
        for k in s:
            k["ts_us"] -= t0
    last_ends = sorted(s[-1]["ts_us"] + s[-1]["dur_us"] for s in by_stream.values())
    small_level = sum(e["dur"] for e in kern if "hash_level_kernel" in e["name"] and (e.get("args", {}).get("grid") or [99])[0] <= 4)
    summary = {
        "card": info["card"], "lanes": lanes, "step_us": t1 - t0, "kernels": len(kern), "streams": len(by_stream),
        "tail_us": last_ends[-1] - last_ends[0] if last_ends else None,
        "small_level_launch_us_summed": small_level, "small_level_launch_share": small_level / (t1 - t0),
        "note": "step_us: first kernel start to last kernel end of the profiled step (profiler on); shares are summed kernel time over the step span (lanes overlap, so shares may add to more than 1)",
    }
    json.dump({k: v for k, v in sorted(by_stream.items())}, open(os.path.join(args.out, "timeline.json"), "w"))
    json.dump(summary, open(os.path.join(args.out, "summary.json"), "w"), indent=1)
    print(json.dumps(summary), flush=True)
    ctx.close()


if __name__ == "__main__":
    main()
