#!/usr/bin/env python3
"""bench.py — headline benchmark of the hot path (BASELINE.json metric: MPT nodes keccak-hashed/sec
and blocks decoded/sec).

  python bench.py --gpus N --steps K --warmup W            this repo's CUDA path, one rank per GPU
  python bench.py --impl reference --gpus N --steps K ...   the reference's CPU algorithm (oracle port)
                                                            on the host cores, same metric and config

Workload (config.workload): C2, the mainnet-shaped block of BASELINE.json configs[1] — ~20k touched
accounts embedded in a virtual 16^7-account state, 200 txns — one block per GPU per step (weak
scaling: rank r decodes the block of seed 2 + r).  A step = every Keccak of the block: all
addresses / slots / code plus every node of every version of the state, storage, txn and receipt
tries, hashed level-synchronously.
  value  nodes/s with the block's arena and key messages already resident in HBM (device time,
         CUDA events on the library's stream, L2 flushed between steps)
  e2e    the same metric through the C ABI (ppd_block_decode) with HOST buffers: FlatBlock in,
         IrDump out, every host<->device copy and all host work inside the timed region
One JSON line on stdout (rank 0).

  --dump-outputs DIR   after the timed steps, write what the last timed step returned to its caller as .npy files
                       (see dump_ir_records); the inputs depend on the arguments alone, so two builds can be compared
                       file for file
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# one CUDA stream per resident block: ask for the 32 hardware queues the device has (8 unless set) before torch creates the context
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ALU_OPS_PER_PERM = 4354  # SURVEY.md 8d: 24 rounds x ~180 LOP3/SHF + 34 to absorb a rate block
ALU_LANES_PER_SM_CLK = 64
N_SM = 148


def load_traffic():
    """Mean DRAM bytes per hash_level_kernel launch from the latest committed ncu launch list (profiles/rNN_traffic.json)."""
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_traffic.json")))
    if not files:
        return None, None
    d = json.load(open(files[-1]))
    return d.get("dram_bytes_per_launch_mean"), os.path.relpath(files[-1], ROOT)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "sm_max_mhz": d.get("sm_max_mhz", 1965.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "source": "fallback"}


class ClockSampler:
    FIELDS = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = str(gpu_index)
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", self.gpu],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True,
            )
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) >= 8:
                self.rows.append(parts)

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if r[4 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


# SURVEY.md 8d's C2: 20k touched accounts in a virtual 16^7-account state, 15 % contracts, 200 txns, ~100 accounts and
# ~150 slot accesses per txn (15 contracts x (0..10 reads + 0..10 writes)), self-destructs.  Departures, stated in
# config.departures: storage tries are witnessed in full (the generator has no hashed-out siblings inside storage tries),
# so slots per contract are log-uniform 1..256 instead of 1..4096; no accounts are created (in a virtual state a new
# address lands on a hashed-out sibling, which the reference rejects).
C2_PARAMS = dict(contract_frac=0.15, slots_lo=1, slots_hi=256, virtual_depth=7, virtual_accounts_log16=7, slot_reads=(0, 10), slot_writes=(0, 10),
                 allow_new_accounts=False, allow_self_destruct=True, inline_code_frac=0.02)
C2_TAG = "r2"  # cache key of the generated blocks: bump when C2_PARAMS change
C2_DEPARTURES = "slots per contract log-uniform 1..256 with storage tries witnessed in full (spec: 1..4096 with hashed siblings); no new accounts"


def c2_block(seed, scale):
    """One synthetic C2 block (SURVEY.md 8d) as a FlatBlock; cached under /tmp."""
    from proof_protocol_decoder_b200 import synth

    cache = f"/tmp/ppd_c2{C2_TAG}_seed{seed}_scale{scale}.flat"
    if os.path.exists(cache):
        return open(cache, "rb").read()
    blk = synth.gen_block(
        seed,
        n_accounts=max(10, int(20000 * scale)),
        n_txns=max(2, int(200 * scale)),
        accounts_per_txn=(80, 120) if scale >= 0.5 else (max(2, int(80 * scale * 4)), max(4, int(120 * scale * 4))),
        **C2_PARAMS,
    )
    f = blk.flat
    try:
        tmp = cache + f".{os.getpid()}.tmp"
        open(tmp, "wb").write(f)
        os.replace(tmp, cache)
    except OSError:
        pass
    return f


def _c2_block_job(a):
    c2_block(*a)
    return 0


def c2_blocks(seeds, scale, procs):
    """The blocks of the given seeds; missing ones are generated in parallel worker processes (the
    generator is pure Python: ~10 s per full-size block)."""
    missing = [s for s in seeds if not os.path.exists(f"/tmp/ppd_c2{C2_TAG}_seed{s}_scale{scale}.flat")]
    if len(missing) > 1 and procs > 1:
        import multiprocessing as mp

        with mp.get_context("fork").Pool(min(procs, len(missing))) as pool:
            pool.map(_c2_block_job, [(s, scale) for s in missing])
    if missing:
        os.sync()  # the cache files (gigabytes of dirty pages) are written back now, not under the timed steps
    return [c2_block(s, scale) for s in seeds]


DUMP_CHUNKS, DUMP_CHUNK, DUMP_SEED = 64, 512, 20250101  # 32 KiB of every IrDump, 128 KiB as float32


def ir_dump_record(view):
    """What --dump-outputs keeps of one IrDump (bytes or a memoryview): its length, its SHA-256 (which covers every byte)
    and DUMP_CHUNKS runs of DUMP_CHUNK bytes at offsets drawn from a fixed seed, so that two dumps of the same length are
    sampled at the same places.  Cheap enough to run on the library's callback thread before the buffer is released."""
    import numpy as np

    a = np.frombuffer(view, dtype=np.uint8)
    n = a.size
    offsets = np.sort((np.random.default_rng(DUMP_SEED).random(DUMP_CHUNKS) * max(n - DUMP_CHUNK, 0)).astype(np.int64))
    idx = offsets[:, None] + np.arange(DUMP_CHUNK)
    sample = np.full(idx.shape, -1.0, dtype=np.float32)  # -1: past the end of a dump shorter than one run
    inside = idx < n
    sample[inside] = a[idx[inside]]
    return n, hashlib.sha256(view).digest(), offsets, sample


def dump_ir_records(out_dir, records):
    """records: one ir_dump_record per block, in the order of the step's input list.  Writes
      ir_dump_nbytes.npy          float64 [blocks]               length of each IrDump
      ir_dump_sha256.npy          float32 [blocks, 32]           its SHA-256, one byte per entry
      ir_dump_sample_offsets.npy  float64 [blocks, CHUNKS]       where each sampled run starts
      ir_dump_sample.npy          float32 [blocks, CHUNKS, CHUNK] the sampled bytes (-1 past the end)"""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {
        "ir_dump_nbytes": np.array([r[0] for r in records], dtype=np.float64),
        "ir_dump_sha256": np.array([list(r[1]) for r in records], dtype=np.float32).reshape(len(records), 32),
        "ir_dump_sample_offsets": np.array([r[2] for r in records], dtype=np.float64).reshape(len(records), DUMP_CHUNKS),
        "ir_dump_sample": np.array([r[3] for r in records], dtype=np.float32).reshape(len(records), DUMP_CHUNKS, DUMP_CHUNK),
    }
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    print(f"bench: wrote {', '.join(arrays)} ({len(records)} blocks) to {out_dir}", file=sys.stderr, flush=True)


def oracle_time_block(flat_bytes, repeats, threads, keep=None):
    """Decode `flat_bytes` `repeats` times on each of `threads` host threads (ctypes releases the GIL).
    Returns (wall seconds, stats of one decode).  With a list as `keep`, the IrDump of the last decode is appended to it."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import ppd_oracle_lib

    oracle = ppd_oracle_lib.load()
    stats = {}

    def work():
        for _ in range(repeats):
            out = oracle.block_decode(flat_bytes)
        stats.update(oracle.last_stats())
        if keep is not None and not keep:
            keep.append(out)

    ts = [threading.Thread(target=work) for _ in range(threads)]
    t0 = time.perf_counter()
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return time.perf_counter() - t0, stats


def run_reference(args, rank, world):
    """The reference's CPU algorithm for the path (the oracle: a C++ port of the reference's Rust, which cannot be
    compiled here) on all host cores, on the SAME config as the b200 arm: every step decodes one full-size C2 block
    per core (about 10 s per block per core; the warm-up is one step).  Rank 0 alone works."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample_scale = args.ref_scale
    flat_bytes = c2_block(2, sample_scale)
    for _ in range(max(1, min(args.warmup, 1))):
        oracle_time_block(flat_bytes, 1, cores)
    t_total, st, last = 0.0, {}, []
    for k in range(args.steps):
        t, st = oracle_time_block(flat_bytes, 1, cores, keep=last if k == args.steps - 1 else None)
        t_total += t
    if args.dump_outputs:
        dump_ir_records(args.dump_outputs, [ir_dump_record(last[0])])
    nodes = st["nodes_hashed"] * cores * args.steps
    value = nodes / t_total
    workload = "C2 mainnet-shaped block (BASELINE.json configs[1])" + ("" if sample_scale == 1.0 else f" at {sample_scale:g}x scale")
    line = {
        "impl": "reference",
        "metric": "mpt_nodes_keccak_hashed_per_sec",
        "value": value,
        "unit": "nodes/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": max(1, min(args.warmup, 1)),
        "ms_per_step": 1e3 * t_total / args.steps,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u64",
        "data": "synthetic",
        "config": {"workload": workload, "scale": sample_scale, "departures": C2_DEPARTURES,
                   "sample": f"one {sample_scale:g}x-scale C2 block (seed 2) per core per step, {cores} cores", "l2": "n/a (CPU)"},
        "blocks_per_sec": cores * args.steps / t_total,
        "nodes_hashed_per_block": st["nodes_hashed"],
        "cpu_baseline": {
            "value": value, "unit": "nodes/s", "cores": cores, "kind": "port",
            "sample": f"one {sample_scale:g}x-scale C2 block ({st['nodes_hashed']} node hashes) per core per step; C++ restatement of the reference algorithm (the Rust reference cannot be built in this image)",
        },
        "e2e": {"value": value, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def c5_sweep(ctx, sizes, peaks, sm_mhz):
    """Config 5: state-trie rehash over sorted leaves already resident in HBM (structure built and
    hashed on the GPU).  Reported beside the headline to show the hashing kernels at scale."""
    import torch

    out = []
    for n in sizes:
        try:
            g = torch.Generator(device="cuda")
            g.manual_seed(5)
            keys = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
            hi = keys[:, :8].to(torch.int64)
            k64 = torch.zeros(n, dtype=torch.int64, device="cuda")
            for b in range(8):
                k64 = (k64 << 8) | hi[:, b]
            order = torch.argsort((k64 >> 1) & 0x7FFFFFFFFFFFFFFF)  # top 63 bits, unsigned order
            del hi, k64
            keys = keys[order].contiguous()
            del order
            lens = torch.randint(70, 81, (n,), dtype=torch.int64, device="cuda", generator=g)
            val_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
            val_off[1:] = torch.cumsum(lens, 0)
            vb = int(val_off[-1].item())
            vals = torch.randint(0, 256, (vb,), dtype=torch.uint8, device="cuda", generator=g)
            torch.cuda.synchronize()
            best = None
            for _ in range(3):
                ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), val_off.data_ptr(), vals.data_ptr(), n, vb)
                st = ctx.stats()
                if best is None or st["gpu_ms"] < best["gpu_ms"]:
                    best = st
            sec = best["gpu_ms"] / 1e3
            alu_peak = ALU_LANES_PER_SM_CLK * N_SM * (sm_mhz or peaks["sm_max_mhz"]) * 1e6
            out.append({
                "leaves": n, "nodes_hashed": best["nodes_hashed"], "permutations": best["node_permutations"], "gpu_ms": best["gpu_ms"],
                "nodes_per_sec": best["nodes_hashed"] / sec, "perms_per_sec": best["node_permutations"] / sec,
                "alu_frac": best["node_permutations"] * ALU_OPS_PER_PERM / sec / alu_peak,
                "hbm_frac": (best["node_bytes"] + 32 * best["nodes_hashed"]) / sec / 1e9 / peaks["hbm_gbs"],
                "note": "includes building the trie structure on the GPU (LCP, branch discovery, counting sort)",
            })
            del keys, vals, val_off, lens
            torch.cuda.empty_cache()
        except Exception as e:  # noqa: BLE001 — the sweep is supplementary; never lose the headline line
            out.append({"leaves": n, "error": str(e)[:200]})
            break
    return out


def _unit_leaves(torch, n, seed, top_nibble, val_lo, val_hi):
    """n sorted leaves on the device whose keys start with `top_nibble` (a deterministic function of the seed, so that
    every world size hashes the same trie)."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    keys = torch.randint(0, 256, (n, 32), dtype=torch.uint8, device="cuda", generator=g)
    keys[:, 0] = (keys[:, 0] & 15) | (top_nibble << 4)
    k64 = torch.zeros(n, dtype=torch.int64, device="cuda")
    for b in range(8):
        k64 = (k64 << 8) | keys[:, b].to(torch.int64)
    order = torch.argsort((k64 >> 1) & 0x7FFFFFFFFFFFFFFF)
    keys = keys[order].contiguous()
    del k64, order
    lens = torch.randint(val_lo, val_hi + 1, (n,), dtype=torch.int64, device="cuda", generator=g)
    val_off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    val_off[1:] = torch.cumsum(lens, 0)
    vb = int(val_off[-1].item())
    vals = torch.randint(1, 256, (vb,), dtype=torch.uint8, device="cuda", generator=g)
    return keys, val_off, vals, vb


def _gather_refs(torch, dist, local, n_units):
    """{unit: 32-byte ref} of every rank -> all refs on every rank (one all-reduce: units are disjoint)."""
    buf = torch.zeros(32 * n_units, dtype=torch.int32, device="cuda")
    for u, r in local.items():
        buf[32 * u: 32 * u + 32] = torch.frombuffer(bytearray(r), dtype=torch.uint8).to("cuda").to(torch.int32)
    if dist is not None:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
    raw = bytes(buf.to(torch.uint8).cpu().numpy().tobytes())
    return [raw[32 * u: 32 * u + 32] for u in range(n_units)]


def split_legs(ctx, torch, dist, rank, world, args, barrier, max_over_ranks, sum_over_ranks, n1):
    """Config 5 (one huge trie) and the storage side of config 3 (a few 1 M-slot tries) over `world` GPUs (SURVEY.md 8e):
    tries are cut at their top nibble into 16 sub-tries, the units are dealt to the ranks, each rank hashes its units
    (structure built and hashed on its GPU), one NCCL all-reduce gathers the 32-byte refs, rank 0 hashes the top
    branches (and, for config 3, the state trie whose account leaves carry the gathered storage roots,
    decoding.rs:438-447).  Strong scaling: the tries are the same for every world size, so are their roots."""
    from proof_protocol_decoder_b200 import synth

    out = {}
    # ---------------- config 5 ----------------
    total = args.c5_leaves
    per = total // 16
    mine = [i for i in range(16) if i % world == rank]
    units = {i: _unit_leaves(torch, per, 5000 + i, i, 70, 80) for i in mine}
    for _ in range(2):  # warm-up (buffers of the context grow to size)
        for i in mine[:1]:
            k, vo, v, vb = units[i]
            ctx.trie_subroot_sorted_leaves_dev(k.data_ptr(), vo.data_ptr(), v.data_ptr(), per, vb, 1)
    barrier()
    t0 = time.perf_counter()
    local, nodes, perms, dev_ms = {}, 0, 0, 0.0
    for i in mine:
        k, vo, v, vb = units[i]
        local[i] = ctx.trie_subroot_sorted_leaves_dev(k.data_ptr(), vo.data_ptr(), v.data_ptr(), per, vb, 1)
        st = ctx.stats()
        nodes += st["nodes_hashed"]
        perms += st["node_permutations"]
        dev_ms += st["gpu_ms"]
    refs = _gather_refs(torch, dist, local, 16)
    root = ctx.trie_root_from_children(b"".join(refs), 0xFFFF) if rank == 0 else b""
    torch.cuda.synchronize()
    wall = max_over_ranks(time.perf_counter() - t0)
    barrier()
    nodes_all, perms_all, dev_ms_max = sum_over_ranks(float(nodes)), sum_over_ranks(float(perms)), max_over_ranks(dev_ms)
    leg = {"leaves": per * 16, "ms": 1e3 * wall, "device_ms_max_over_ranks": dev_ms_max, "nodes_hashed": nodes_all + 1, "nodes_per_sec": (nodes_all + 1) / wall,
           "permutations_per_sec": perms_all / wall, "root": root.hex() if rank == 0 else None, "units_per_rank": len(mine),
           "note": "16 sub-tries by top nibble dealt to the ranks; refs gathered by one NCCL all-reduce of 512 bytes; top branch on rank 0; wall clock between barriers, max over ranks"}
    if world == 1:
        # the same trie hashed whole: the split must give its root
        keys = torch.cat([units[i][0] for i in range(16)])
        lens = torch.cat([units[i][1][1:] - units[i][1][:-1] for i in range(16)])
        val_off = torch.zeros(per * 16 + 1, dtype=torch.int64, device="cuda")
        val_off[1:] = torch.cumsum(lens, 0)
        vals = torch.cat([units[i][2] for i in range(16)])
        whole = ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), val_off.data_ptr(), vals.data_ptr(), per * 16, int(val_off[-1].item()))
        leg["whole_trie_ms"] = ctx.stats()["gpu_ms"]
        leg["equals_whole_trie_root"] = whole == root
        del keys, lens, val_off, vals
    elif rank == 0 and n1.get("c5_split"):
        leg["root_equals_n1_run"] = n1["c5_split"].get("root") == leg["root"]
        leg["speedup_vs_n1"] = n1["c5_split"]["ms"] / leg["ms"]
        leg["efficiency_vs_n1"] = leg["speedup_vs_n1"] / world
    out["c5_split"] = leg
    del units
    torch.cuda.empty_cache()
    # ---------------- config 3: storage tries sharded, roots joined into the account leaves ----------------
    n_c, slots = 4, args.c3_slots
    per = slots // 16
    all_units = [(c, i) for c in range(n_c) for i in range(16)]
    mine = [u for k, u in enumerate(all_units) if k % world == rank]
    units = {u: _unit_leaves(torch, per, 3000 + 16 * u[0] + u[1], u[1], 1, 33) for u in mine}
    barrier()
    t0 = time.perf_counter()
    local, nodes, perms = {}, 0, 0
    for (c, i) in mine:
        k, vo, v, vb = units[(c, i)]
        local[16 * c + i] = ctx.trie_subroot_sorted_leaves_dev(k.data_ptr(), vo.data_ptr(), v.data_ptr(), per, vb, 1)
        st = ctx.stats()
        nodes += st["nodes_hashed"]
        perms += st["node_permutations"]
    refs = _gather_refs(torch, dist, local, 16 * n_c)
    state_root = b""
    if rank == 0:
        storage_roots = [ctx.trie_root_from_children(b"".join(refs[16 * c: 16 * c + 16]), 0xFFFF) for c in range(n_c)]
        # the state trie: 1 000 plain accounts + the contracts, whose leaves carry the storage roots just gathered
        import numpy as np

        rng = np.random.default_rng(3)
        n_acc = 1000 + n_c
        hk = rng.bytes(32 * n_acc)
        items = []
        for a in range(n_acc):
            sroot = storage_roots[a] if a < n_c else bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")
            rlp = synth.rlp_list([synth.rlp_int(a + 1), synth.rlp_int(10 ** 18 + a), synth.rlp_str(sroot), synth.rlp_str(hk[32 * a: 32 * a + 32][::-1])])
            items.append((hk[32 * a: 32 * a + 32], rlp))
        items.sort()
        keys = np.frombuffer(b"".join(k for k, _ in items), dtype=np.uint8).reshape(-1, 32)
        val_off = np.zeros(n_acc + 1, dtype=np.uint64)
        val_off[1:] = np.cumsum([len(v) for _, v in items])
        vals = np.frombuffer(b"".join(v for _, v in items), dtype=np.uint8)
        state_root = ctx.trie_root_sorted_leaves(keys, val_off, vals)
        nodes += ctx.stats()["nodes_hashed"] + n_c
    torch.cuda.synchronize()
    wall = max_over_ranks(time.perf_counter() - t0)
    barrier()
    nodes_all = sum_over_ranks(float(nodes))
    leg = {"contracts": n_c, "slots_per_contract": per * 16, "plain_accounts": 1000, "ms": 1e3 * wall, "nodes_hashed": nodes_all, "nodes_per_sec": nodes_all / wall,
           "state_root": state_root.hex() if rank == 0 else None, "units_per_rank": len(mine),
           "note": "64 storage sub-tries (4 contracts x 16 top nibbles) dealt to the ranks; their refs gathered by one NCCL all-reduce; rank 0 hashes the 4 top branches and the state trie whose account leaves carry those storage roots"}
    if world > 1 and rank == 0 and n1.get("c3_sharded"):
        leg["state_root_equals_n1_run"] = n1["c3_sharded"].get("state_root") == leg["state_root"]
        leg["speedup_vs_n1"] = n1["c3_sharded"]["ms"] / leg["ms"]
        leg["efficiency_vs_n1"] = leg["speedup_vs_n1"] / world
    out["c3_sharded"] = leg
    del units
    torch.cuda.empty_cache()
    return out


def measure_pcie(torch, mb=64, secs=0.3, barrier=None):
    """Pinned-memory copy bandwidth of this GPU's link, both directions at once (GB/s in the slower direction), measured
    for `secs` on several streams while every other rank does the same (the ranks start together behind `barrier`): GPUs
    of one box may share a PCIe switch or root port, and what bounds a pipeline that streams FlatBlocks in and IrDumps
    out is what the link gives when all of them copy."""
    n = mb << 20
    k = 4
    h_in = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(k)]
    h_out = [torch.empty(n, dtype=torch.uint8).pin_memory() for _ in range(k)]
    d_in = [torch.empty(n, dtype=torch.uint8, device="cuda") for _ in range(k)]
    d_out = [torch.empty(n, dtype=torch.uint8, device="cuda") for _ in range(k)]
    s_up = [torch.cuda.Stream() for _ in range(k)]
    s_dn = [torch.cuda.Stream() for _ in range(k)]
    for i in range(k):  # touch everything once
        d_in[i].copy_(h_in[i], non_blocking=True)
        h_out[i].copy_(d_out[i], non_blocking=True)
    torch.cuda.synchronize()
    if barrier is not None:
        barrier()
    t0 = time.perf_counter()
    rounds = 0
    while time.perf_counter() - t0 < secs:
        for i in range(k):
            with torch.cuda.stream(s_up[i]):
                d_in[i].copy_(h_in[i], non_blocking=True)
            with torch.cuda.stream(s_dn[i]):
                h_out[i].copy_(d_out[i], non_blocking=True)
        torch.cuda.synchronize()
        rounds += 1
    dt = time.perf_counter() - t0
    return rounds * k * n / dt / 1e9


N1_CACHE = "/tmp/ppd_bench_n1.json"  # the N=1 run leaves its e2e blocks/s and the oracle's node count here for the N>1 runs of the same box


def run_b200(args, rank, world, local_rank):
    cores = os.cpu_count() or 1
    n_blocks = min(64, args.blocks_per_step or 64)  # per GPU, whatever the world size (weak scaling); the library keeps up to 64 lanes resident
    # one host thread per resident block: with the txn loop on the device a block's thread mostly waits for its lane
    os.environ.setdefault("PPD_HOST_THREADS", str(n_blocks))
    threads = int(os.environ["PPD_HOST_THREADS"])
    seeds = [2 + rank * n_blocks + j for j in range(n_blocks)]
    # generated before CUDA is touched (worker processes are forked); ranks generate their own blocks
    flats = c2_blocks(seeds, args.scale, max(1, cores // world))
    flat_total = sum(len(f) for f in flats)

    import torch

    from proof_protocol_decoder_b200.lib import Context

    peaks = load_peaks()
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
        # this rank's threads on its share of the host cores (the ranks of a box share them)
        try:
            avail = sorted(os.sched_getaffinity(0))
            share = max(1, len(avail) // world)
            os.sched_setaffinity(0, set(avail[local_rank * share:(local_rank + 1) * share] or avail))
        except (AttributeError, OSError):
            pass

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    ctx = Context(local_rank)
    pcie_gbs = measure_pcie(torch, barrier=barrier)  # (all ranks at once)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2
    # the step's inputs live in page-locked host memory (ppd_alloc_pinned), as a caller that serialises its
    # BlockTrace for the library would place them; every step copies them to the device again
    flats = [ctx.pinned_copy(f) for f in flats]

    # a timed end-to-end step decodes every block e2e_mult times in one call (512 blocks by default): the pipeline's ramp
    # at both ends of a call (one block's latency in flight, ~70 ms) is then a small share, as in a node that keeps feeding
    # blocks; outputs are consumed as they finish, so only those in flight are held
    e2e_mult = max(1, args.e2e_mult)

    def decode_step(mult=1, records=None):
        # ppd_blocks_decode_stream: every block's IrDump is handed over (and read, and released) as soon as it is done;
        # with `records`, the first decode of every distinct block also leaves its ir_dump_record there
        got = []

        def on_done(i, o):
            if isinstance(o, Exception):
                raise o
            if records is not None and i < len(flats):
                records[i] = ir_dump_record(o.view)
            got.append(o.nbytes + o.view[0] + o.view[o.nbytes - 1])  # read the result
            o.close()

        ctx.blocks_decode_stream(flats * mult, on_done)
        assert len(got) == len(flats) * mult
        return sum(got)

    # ---- warm-up (also leaves the arenas resident for the device-resident measurements) ----
    for _ in range(max(3, args.warmup)):
        ir_len = decode_step(e2e_mult)  # (the size of the timed calls: their page-locked output buffers are made here)
    st = ctx.stats()
    on_device = int(st["txn_loops_on_gpu"])
    # the blocks a replay covers: the last block of every lane is what stays resident in HBM
    resident = ctx.replay_lanes()

    def replay(what):
        """device time per step of the selected stages, every lane replaying them concurrently on resident data"""
        for _ in range(max(3, args.warmup)):
            ctx.replay_last(what)
        barrier()
        ms = 0.0
        for _ in range(args.steps):
            flush.zero_()
            torch.cuda.synchronize()
            ms += ctx.replay_last(what)
        barrier()
        return max_over_ranks(ms) / args.steps

    sampler = ClockSampler(local_rank)
    sampler.start()
    hash_ms = replay(ctx.REPLAY_HASH)
    parse_ms = replay(ctx.REPLAY_PARSE) if st["witnesses_on_gpu"] else 0.0
    txn_ms = replay(ctx.REPLAY_TXN) if on_device else 0.0
    dump_ms = replay(ctx.REPLAY_DUMP) if on_device else 0.0
    all_ms = replay(ctx.REPLAY_ALL)
    # ---- end to end through the C ABI with host buffers ----
    # (--dump-outputs: rank 0 records the last step's IrDumps; hashing them adds host work to that step alone)
    records = {} if args.dump_outputs and rank == 0 else None
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        ir_len = decode_step(e2e_mult, records if k == args.steps - 1 else None)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    e2e_s = max_over_ranks(e2e_s)
    if records is not None:
        dump_ir_records(args.dump_outputs, [records[j] for j in range(n_blocks)])
    clocks = sampler.stop()
    st = ctx.stats()
    # latency of one block alone, and the node count of the seed-2 block (rank 0) for the normalisation below
    single = []
    for _ in range(3):
        t1 = time.perf_counter()
        with ctx.block_decode_view(flats[0]) as v:
            _ = v.view[0]
        single.append(time.perf_counter() - t1)
    own_nodes_block0 = ctx.stats()["nodes_hashed"]

    nodes_all = sum_over_ranks(float(st["nodes_hashed"]))
    perms_all = sum_over_ranks(float(st["node_permutations"] + st["key_permutations"]))
    keys_all = sum_over_ranks(float(st["key_hashes"]))
    host_busy_all = sum_over_ranks(float(st["host_busy_ms"]))
    blocks_step = n_blocks * e2e_mult  # blocks of one end-to-end step on this GPU (the stats of the last call cover them)
    dev_s_per_step = hash_ms / 1e3
    e2e_s_per_step = e2e_s / args.steps
    sm_mhz = clocks.get("sm_mhz")
    alu_peak = ALU_LANES_PER_SM_CLK * N_SM * (sm_mhz or peaks["sm_max_mhz"]) * 1e6  # instr/s on one GPU
    algo_bytes = st["node_bytes"] + 32 * st["nodes_hashed"]  # SURVEY.md 8d: L + 32 per hashed node (this rank)
    achieved_gbs = algo_bytes * (resident / blocks_step) / dev_s_per_step / 1e9
    traffic, traffic_src = load_traffic()
    level_launches = max(1, int(st["level_launches"]))
    wit_bytes_all = sum_over_ranks(float(st["witness_bytes"]))
    wit_ins_all = sum_over_ranks(float(st["witness_instructions"]))
    blocks_all = world * blocks_step
    h2d_all, d2h_all = sum_over_ranks(float(st["h2d_bytes"])), sum_over_ranks(float(st["d2h_bytes"]))
    e2e_bps = blocks_all / e2e_s_per_step
    # ---- the reference's node count for the same block (its hashing work is the unit both arms are quoted in) ----
    cpu_baseline, oracle_nodes = None, None
    if rank == 0 and world == 1:
        sample = c2_block(2, args.ref_scale)
        t, ost = oracle_time_block(sample, 1, 1)
        cpu_baseline = {
            "value": ost["nodes_hashed"] / t,
            "unit": "nodes/s",
            "cores": 1,
            "kind": "port",
            "blocks_per_sec": 1.0 / t,
            "nodes_hashed_per_block": ost["nodes_hashed"],
            "sample": f"one {args.ref_scale:g}x-scale C2 block (seed 2: {ost['nodes_hashed']} node hashes, {t:.2f} s) on 1 core; C++ restatement of the reference algorithm (the Rust reference cannot be built in this image)",
        }
        if args.ref_scale == args.scale:
            oracle_nodes = ost["nodes_hashed"]
    n1 = {}
    if world == 1 and rank == 0:
        n1 = {"e2e_blocks_per_sec": e2e_bps, "oracle_nodes_block0": oracle_nodes, "own_nodes_block0": own_nodes_block0, "scale": args.scale, "tag": C2_TAG}
        try:
            json.dump(n1, open(N1_CACHE, "w"))
        except OSError:
            pass
    elif os.path.exists(N1_CACHE):
        try:
            n1 = json.load(open(N1_CACHE))
            if n1.get("scale") != args.scale or n1.get("tag") != C2_TAG:
                n1 = {}
        except (OSError, ValueError):
            n1 = {}
    norm = 1.0
    if n1.get("oracle_nodes_block0") and n1.get("own_nodes_block0"):
        norm = n1["oracle_nodes_block0"] / n1["own_nodes_block0"]
    # ---- what bounds end-to-end blocks/s ----
    per_block_host_ms = host_busy_all / blocks_all
    per_block_h2d, per_block_d2h = h2d_all / blocks_all, d2h_all / blocks_all
    blocks_replayed = world * resident
    bounds = {
        "device_pipeline": blocks_replayed / ((hash_ms + parse_ms + dump_ms) / 1e3),
        "pcie": sum_over_ranks(pcie_gbs) * 1e9 / max(per_block_h2d, per_block_d2h),
        "host_cores": cores / (per_block_host_ms / 1e3) if per_block_host_ms else None,
    }
    limiter = min((k for k in bounds if bounds[k]), key=lambda k: bounds[k])
    line = {
        "metric": "mpt_nodes_keccak_hashed_per_sec",
        "value": norm * nodes_all * (resident / blocks_step) / dev_s_per_step,
        "unit": "nodes/s",
        "n_gpus": world,
        "steps": args.steps,
        "warmup": max(3, args.warmup),
        "ms_per_step": 1e3 * dev_s_per_step,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "u64",
        "data": "synthetic",
        "config": {
            "workload": f"C2 mainnet-shaped blocks (BASELINE.json configs[1]): 20k touched accounts in a virtual 16^7-account state, 200 txns each; a batch of {n_blocks} independent blocks per GPU per step, one lane (stream + pools) per block, {threads} host thread(s) per GPU",
            "scale": args.scale,
            "departures": C2_DEPARTURES,
            "blocks_per_step_per_gpu": blocks_step,
            "distinct_blocks_per_gpu": n_blocks,
            "host_threads_per_gpu": threads,
            "host_cores": cores,
            "flat_block_bytes_per_step": flat_total * e2e_mult,
            "ir_dump_bytes_per_step": ir_len,
            "arena_nodes": st["arena_nodes"],
            "levels": st["levels"],
            "txn_loops_on_device_per_step": int(st["txn_loops_on_gpu"]),
            "l2": "flushed between timed device-resident steps (256 MiB write)",
            "parallelism": f"blocks sharded over {world} GPU(s), no data-path collective",
        },
        "value_note": "node hashes per second of the hashing kernels (key hashing + both level sweeps of every block, lanes concurrent) on arenas resident in HBM, in units of the REFERENCE's node hashes for the same block (nodes_normalisation)",
        "nodes_normalisation": {"factor": norm, "oracle_nodes_block0": n1.get("oracle_nodes_block0"), "own_nodes_block0": n1.get("own_nodes_block0"),
                                "note": "the library hashes every node of every trie version it builds; the reference hashes a few per cent fewer or more (it never builds unobserved versions, but hashes per-txn subsets): throughputs are quoted in the reference's count"},
        "blocks_per_sec": blocks_replayed / (all_ms / 1e3),
        "blocks_per_sec_note": "device-resident: the blocks of a step / device time of the WHOLE pipeline replayed on resident data (witness parse, key hashing, pre-image sweep, by-root join, txn loop, second sweep, IR sizing and emit), every lane in pipeline order, lanes concurrent",
        "device_ms_per_step": {"hashing": hash_ms, "parse": parse_ms, "txn_loop": txn_ms, "dump": dump_ms, "whole_pipeline": all_ms, "blocks_replayed": blocks_replayed,
                               "note": "each stage replayed alone with all lanes concurrent (the resident block of every lane), then all of them together"},
        "blocks_per_sec_hashing_only": blocks_replayed / dev_s_per_step,
        "permutations_per_sec": perms_all * (resident / blocks_step) / dev_s_per_step,
        "nodes_hashed_per_step": nodes_all,
        "key_hashes_per_step": keys_all,
        "e2e": {
            "value": norm * nodes_all / e2e_s_per_step,
            "unit": "nodes/s",
            "blocks_per_sec": e2e_bps,
            "ms_per_step": 1e3 * e2e_s_per_step,
            "single_block_latency_ms": 1e3 * min(single),
            "h2d_bytes_per_step": h2d_all,
            "d2h_bytes_per_step": d2h_all,
            "boundary_bytes_per_step": {"flat_blocks": flat_total * e2e_mult * world, "ir_dumps": ir_len * world},
            "host_busy_ms_per_block": per_block_host_ms,
            "note": "ppd_blocks_decode_stream: FlatBlocks (page-locked host memory) -> IrDumps (page-locked host memory, read and released by the callback as each block finishes); every host<->device copy and all host work (flat input reading, descriptor tables, launches) inside the timed region",
        },
        "e2e_blocks_per_sec": e2e_bps,
        "e2e_efficiency_vs_n1": (e2e_bps / (world * n1["e2e_blocks_per_sec"])) if n1.get("e2e_blocks_per_sec") else None,
        "limiter": {
            "name": limiter,
            "bounds_blocks_per_sec": bounds,
            "pcie_gbs_per_direction": pcie_gbs,
            "pcie_gbs_per_direction_all_gpus": sum_over_ranks(pcie_gbs),
            "pcie_bytes_per_block": {"h2d": per_block_h2d, "d2h": per_block_d2h},
            "host_busy_ms_per_block": per_block_host_ms,
            "device_pipeline_lockstep": blocks_replayed / (all_ms / 1e3),
            "note": "upper bounds on end-to-end blocks/s: device_pipeline = the kernels that fill the device (witness parse, key hashing and both level sweeps, IR sizing and emit), each stage replayed by all resident lanes at once, times added; the txn loops run beside them, one SM each (device_pipeline_lockstep: every lane replaying its whole pipeline from the same instant, loops included: stages of different lanes do not overlap there as they do in a running pipeline); pcie = the pinned-copy rate of all GPUs' links measured while every rank copies in both directions at once (GPUs of a box may share a switch or root port), over the bytes a block moves in the busier direction; host_cores = the box's cores over the CPU time a block costs its host thread",
        },
        "gpu_launches": int(st["kernel_launches"]) * args.steps,
        "clocks": clocks,
        "roofline": {
            "bound": "alu",
            "kernel": "hash_level_kernel + keccak256_batch_kernel (all level launches of the batch, lanes concurrent)",
            "achieved": (st["node_permutations"] + st["key_permutations"]) * (resident / blocks_step) * ALU_OPS_PER_PERM / dev_s_per_step / 1e12,
            "peak": alu_peak / 1e12,
            "unit": "Tinstr/s",
            "frac": (st["node_permutations"] + st["key_permutations"]) * (resident / blocks_step) * ALU_OPS_PER_PERM / dev_s_per_step / alu_peak,
            "traffic": traffic,
            "traffic_source": traffic_src,
            "model": f"{ALU_OPS_PER_PERM} ALU-pipe (LOP3/SHF) instructions per keccak-f[1600] permutation (SURVEY.md 8d); peak = {ALU_LANES_PER_SM_CLK} lanes/clk/SM x {N_SM} SMs x SM clock sampled under load",
            "peak_source": "profiles/r02_microbench.txt: dependent-free LOP3/SHF issue measured at 64 lanes/clk/SM (MEASURED_PEAKS.json has no integer peak)",
            "launches_per_step": level_launches,
            "note": "Keccak is bound by the integer ALU pipe, not HBM (SURVEY.md 8d); the HBM view is in roofline_hbm",
        },
        "roofline_hbm": {
            "bound": "hbm",
            "achieved": achieved_gbs,
            "peak": peaks["hbm_gbs"],
            "unit": "GB/s",
            "frac": achieved_gbs / peaks["hbm_gbs"],
            "algorithmic_bytes_per_launch": algo_bytes / level_launches,
            "peak_source": peaks["source"],
            "note": "achieved = sum over the step's level launches of (L + 32) bytes per hashed node / device time of the step",
        },
        "parse": {
            "kernels": "ppd_parse.cu: tile_exit (lists of opcode bytes) / group_exit / top_chain / tile_entry / tile_mark_thin / scans / link (8-wide pyramid level) / shape / emit + emit_keyed / climb (all lanes concurrent)",
            "witnesses_on_gpu_per_step": int(sum_over_ranks(float(st["witnesses_on_gpu"]))),
            "witness_bytes_per_step": wit_bytes_all,
            "instructions_per_step": wit_ins_all,
            "ms_per_step": parse_ms,
            "bound": "hbm",
            "achieved": (7.0 * wit_bytes_all * (resident / blocks_step) / world / (parse_ms / 1e3) / 1e9) if parse_ms else None,
            "peak": peaks["hbm_gbs"],
            "unit": "GB/s",
            "frac": (7.0 * wit_bytes_all * (resident / blocks_step) / world / (parse_ms / 1e3) / 1e9 / peaks["hbm_gbs"]) if parse_ms else None,
            "instructions_per_sec": (wit_ins_all * (resident / blocks_step) / (parse_ms / 1e3)) if parse_ms else None,
            "note": "algorithmic bytes = 7 per witness byte for the boundary search (read the byte, write and re-read its 4-byte exit link, write its 2-byte step link)",
        },
        "txn_loop": {
            "kernels": "ppd_txn.cu: join / acct_claim / prep_* / txn_loop_kernel (one thread block per block of txns; lanes concurrent)",
            "ms_per_step": txn_ms,
            "blocks_per_sec": (blocks_replayed / (txn_ms / 1e3)) if txn_ms else None,
            "bound": "latency (dependent loads down the tries; one resident CTA per block)",
        },
        "dump": {
            "kernels": "ppd_dump.cu: ir_size_kernel + ir_emit_kernel (one thread block per IR)",
            "ms_per_step": dump_ms,
            "bytes_replayed": ir_len * resident / blocks_step,
            "achieved": (ir_len * (resident / blocks_step) / (dump_ms / 1e3) / 1e9) if dump_ms else None,
            "unit": "GB/s written",
            "frac_of_hbm": (ir_len * (resident / blocks_step) / (dump_ms / 1e3) / 1e9 / peaks["hbm_gbs"]) if dump_ms else None,
            "frac_of_pcie": (ir_len * (resident / blocks_step) / (dump_ms / 1e3) / 1e9 / pcie_gbs) if dump_ms else None,
        },
    }
    if not args.no_split:
        try:
            legs = split_legs(ctx, torch, dist, rank, world, args, barrier, max_over_ranks, sum_over_ranks, n1)
            line.update(legs)
            if world == 1 and rank == 0:
                n1.update({k: {"ms": v["ms"], "root": v.get("root"), "state_root": v.get("state_root")} for k, v in legs.items()})
                try:
                    json.dump(n1, open(N1_CACHE, "w"))
                except OSError:
                    pass
        except Exception as e:  # noqa: BLE001 — supplementary legs never cost the headline line
            line["split_legs_error"] = str(e)[:300]
    if cpu_baseline:
        line["cpu_baseline"] = cpu_baseline
    if rank == 0 and world == 1 and not args.no_sweep:
        line["c5_sweep"] = c5_sweep(ctx, [int(x) for x in args.sweep.split(",") if x], peaks, sm_mhz)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark writes nothing there, bytecode included
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="fraction of the C2 block size (1.0 = the named config)")
    ap.add_argument("--blocks-per-step", type=int, default=0, help="blocks per GPU per step (default 64, at most 64)")
    ap.add_argument("--e2e-mult", type=int, default=8, help="an end-to-end step decodes every block this many times in one call")
    ap.add_argument("--ref-scale", type=float, default=1.0, help="size of the CPU arm's block (1.0 = the same config as the b200 arm)")
    ap.add_argument("--sweep", default="1000000,10000000", help="config-5 leaf counts measured beside the headline at N=1")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--c5-leaves", type=int, default=32_000_000, help="leaves of the config-5 trie that is split over the GPUs")
    ap.add_argument("--c3-slots", type=int, default=1_000_000, help="slots of each of the four config-3 storage tries that are sharded over the GPUs")
    ap.add_argument("--no-split", action="store_true", help="skip the c5_split / c3_sharded legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the IrDumps the last end-to-end step returned (length, SHA-256 and a "
                         "fixed sample of each distinct block's dump) to DIR as .npy files; rank 0's blocks only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
