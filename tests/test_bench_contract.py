"""bench.py's output contract, as far as it can be checked without a GPU: the reference arm (`--impl reference`, the
CPU restatement of the reference on the host cores) prints one JSON line with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-scale", "0.02"],
                         capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "mpt_nodes_keccak_hashed_per_sec" and d["unit"] == "nodes/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    return out


def _check_dump(d, n_blocks, flat_blocks, oracle):
    """The files of --dump-outputs: float32/float64 arrays, at most 64 MB in all, whose records are the oracle's IrDumps."""
    import hashlib

    import bench

    names = ["ir_dump_nbytes", "ir_dump_sha256", "ir_dump_sample_offsets", "ir_dump_sample"]
    assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in names)
    assert sum(os.path.getsize(os.path.join(d, n + ".npy")) for n in names) <= 64 << 20
    got = {n: np.load(os.path.join(d, n + ".npy")) for n in names}
    assert all(a.dtype in (np.float32, np.float64) and a.shape[0] == n_blocks for a in got.values())
    for j, fb in enumerate(flat_blocks):
        ir = oracle.block_decode(fb)
        want = bench.ir_dump_record(ir)
        assert got["ir_dump_nbytes"][j] == want[0] == len(ir)
        assert bytes(got["ir_dump_sha256"][j].astype(np.uint8)) == want[1] == hashlib.sha256(ir).digest()
        assert np.array_equal(got["ir_dump_sample_offsets"][j], want[2]) and np.array_equal(got["ir_dump_sample"][j], want[3])
    return got


def test_reference_arm_dumps_the_oracles_ir_dump(tmp_path, oracle):
    """--dump-outputs on the reference arm: the seed-2 block's IrDump, the same for any number of steps."""
    import bench

    for steps in ("1", "2"):
        _bench("--impl", "reference", "--steps", steps, "--warmup", "1", "--ref-scale", "0.02", "--dump-outputs", str(tmp_path / steps))
    a = _check_dump(str(tmp_path / "1"), 1, [bench.c2_block(2, 0.02)], oracle)
    b = _check_dump(str(tmp_path / "2"), 1, [bench.c2_block(2, 0.02)], oracle)
    assert all(np.array_equal(a[k], b[k]) for k in a)


@pytest.mark.gpu
def test_b200_arm_dumps_what_its_last_step_returned(tmp_path, oracle):
    """--dump-outputs on the CUDA arm (a tiny run): one record per distinct block of the step, each the oracle's IrDump of
    that block, identical from run to run."""
    import bench

    small = ["--scale", "0.02", "--ref-scale", "0.02", "--blocks-per-step", "3", "--e2e-mult", "2", "--no-sweep", "--no-split", "--warmup", "1"]
    for run, steps in (("a", "2"), ("b", "1")):
        out = _bench(*small, "--steps", steps, "--dump-outputs", str(tmp_path / run))
        line = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == int(steps)
    flats = [bench.c2_block(2 + j, 0.02) for j in range(3)]
    a = _check_dump(str(tmp_path / "a"), 3, flats, oracle)
    b = _check_dump(str(tmp_path / "b"), 3, flats, oracle)
    assert all(np.array_equal(a[k], b[k]) for k in a)


def test_bench_defaults_name_the_headline_config():
    """The default run is config 2 of BASELINE.json on one GPU with K/W that finish within minutes."""
    sys.path.insert(0, ROOT)
    import bench

    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'add_argument("--gpus", type=int, default=1)' in src
    assert 'add_argument("--steps", type=int, default=5)' in src and 'add_argument("--warmup", type=int, default=3)' in src
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert "20k touched accounts" in baseline["configs"][1] and bench.C2_PARAMS  # the generator parameters of that config
