"""Direct pre-images (FlatBlock kind 2) on the device txn loop, with the by-address storage join.

A Separate{Direct} pre-image is re-spelled as a compact witness on the host (csrc/host_direct.cu) and then takes the same
device path as a witness: GPU parse, key hashing, the txn loop, the IR dump.  What differs is the storage join: the
map of a direct pre-image is keyed by hashed address (csrc/txn_core.h: join_addr_insert / join_addr_resolve), not by
storage root.  An account outside the map has no trie even when its root is that of a trie in the map, and two accounts
with identical tries each keep their own (the by-root join of a Combined pre-image would share one and hand the block
to the host path).

CPU: tests/cpp/direct_loop_check.cpp runs the host path and the device loop on host memory, and checks the join's arrays
entry by entry against the host path's storage map.  GPU: the product equals the oracle byte for byte, on the device
loop, and equals the host path (PPD_HOST_TXN=1)."""
import copy
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from proof_protocol_decoder_b200 import flat, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "proof_protocol_decoder_b200", "csrc")
EMPTY_TRIE = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")


# ---------------------------------------------------------------------------------------------- building blocks
def _rlp_list_items(b: bytes):
    """The byte strings of an RLP list of strings (an account leaf's value)."""

    def item(p):
        x = b[p]
        if x < 0x80:
            return b[p : p + 1], p + 1
        if x < 0xB8:
            return b[p + 1 : p + 1 + x - 0x80], p + 1 + x - 0x80
        k = x - 0xB7
        n = int.from_bytes(b[p + 1 : p + 1 + k], "big")
        return b[p + 1 + k : p + 1 + k + n], p + 1 + k + n

    x = b[0]
    assert x >= 0xC0
    if x < 0xF8:
        p, end = 1, 1 + x - 0xC0
    else:
        k = x - 0xF7
        p = 1 + k
        end = p + int.from_bytes(b[1 : 1 + k], "big")
    out = []
    while p < end:
        s, p = item(p)
        out.append(s)
    return out


def _rlp_str(s: bytes) -> bytes:
    if len(s) == 1 and s[0] < 0x80:
        return s
    if len(s) < 56:
        return bytes([0x80 + len(s)]) + s
    ln = len(s).to_bytes((len(s).bit_length() + 7) // 8, "big")
    return bytes([0xB7 + len(ln)]) + ln + s


def _rlp_list(items) -> bytes:
    body = b"".join(_rlp_str(s) for s in items)
    if len(body) < 56:
        return bytes([0xC0 + len(body)]) + body
    ln = len(body).to_bytes((len(body).bit_length() + 7) // 8, "big")
    return bytes([0xF7 + len(ln)]) + ln + body


def _haddr(nibs):
    nibs = [0] * (64 - len(nibs)) + list(nibs)
    return bytes((nibs[2 * i] << 4) | nibs[2 * i + 1] for i in range(32))


def _accounts(state):
    """hashed address -> [nonce, balance, storage root, code hash] of every account leaf of a direct state trie"""
    out = {}

    def walk(node, path):
        k = node[0]
        if k == "branch":
            for i, c in enumerate(node[1]):
                walk(c, path + [i])
        elif k == "extension":
            walk(node[2], path + list(node[1]))
        elif k == "leaf":
            out[_haddr(path + list(node[1]))] = _rlp_list_items(bytes(node[2]))

    walk(state, [])
    return out


def _with_storage_root(state, haddr, root):
    """the state trie with the storage-root field of one account replaced"""

    def walk(node, path):
        k = node[0]
        if k == "branch":
            return ("branch", [walk(c, path + [i]) for i, c in enumerate(node[1])], node[2])
        if k == "extension":
            return ("extension", node[1], walk(node[2], path + list(node[1])))
        if k == "leaf" and _haddr(path + list(node[1])) == haddr:
            f = _rlp_list_items(bytes(node[2]))
            f[2] = root
            return ("leaf", node[1], _rlp_list(f))
        return node

    return walk(state, [])


def _direct(oracle, blk_flat):
    """(state, storage) of a Combined FlatBlock's tries as direct nodes"""
    return flat.parse_direct_pre_image(oracle.compact_to_direct(flat.pre_image_of(blk_flat)[1]))


def _kind2(blk_flat, state, storage):
    return flat.with_pre_image(blk_flat, flat.PRE_IMAGE_DIRECT, flat.encode_direct_pre_image(state, storage))


def _combined(lib, blk_flat, state, storage):
    return flat.with_pre_image(blk_flat, flat.PRE_IMAGE_COMBINED, lib.direct_to_compact(flat.encode_direct_pre_image(state, storage)))


def _touched(oracle, blk):
    """hashed address -> set of txn indices whose traces touch it"""
    out = {}
    for ti, t in enumerate(blk.txns):
        for addr, _ in t["traces"]:
            out.setdefault(oracle.keccak256(addr), set()).add(ti)
    return out


def _accessed(oracle, blk):
    """hashed addresses whose slots some txn reads or writes"""
    out = set()
    for t in blk.txns:
        for addr, tr in t["traces"]:
            if tr.get("storage_read") or tr.get("storage_written"):
                out.add(oracle.keccak256(addr))
    return out


def _witness_like(oracle, blk, rng):
    """every storage trie cut to the paths of the slots the txns read or write, the rest hashed out (as a real witness
    carries them)"""

    def nibs_of(h):
        return [x for byte in h for x in (byte >> 4, byte & 15)]

    def prune(node, keys):
        if not keys:
            return node if node[0] in ("empty", "hash") else ("hash", bytes(rng.bytes(32)))
        if node[0] == "branch":
            return ("branch", [prune(c, [k[1:] for k in keys if k and k[0] == i]) for i, c in enumerate(node[1])], node[2])
        if node[0] == "extension":
            n = len(node[1])
            return ("extension", node[1], prune(node[2], [k[n:] for k in keys if k[:n] == list(node[1])]))
        return node

    state, storage = _direct(oracle, blk.flat)
    keys = {}
    for t in blk.txns:
        for addr, tr in t["traces"]:
            ks = keys.setdefault(oracle.keccak256(addr), [])
            ks += [nibs_of(oracle.keccak256(s)) for s in tr.get("storage_read") or []]
            ks += [nibs_of(oracle.keccak256(k)) for k, _ in tr.get("storage_written") or []]
    for h, trie in list(storage.items()):
        if keys.get(h):
            storage[h] = prune(trie, keys[h])
    return state, storage


def _shared_tries(oracle, seed):
    """Two accounts a txn touches, both in the map with IDENTICAL storage tries (same root)."""
    blk = synth.gen_block(seed, n_accounts=60, n_txns=4, inline_code_frac=0.0, contract_frac=0.8, slots_lo=4, slots_hi=30, accounts_per_txn=(3, 8))
    state, storage = _direct(oracle, blk.flat)
    acc = _accounts(state)
    for t in blk.txns:
        hs = [oracle.keccak256(a) for a, _ in t["traces"]]
        hs = [h for h in dict.fromkeys(hs) if h in storage and storage[h][0] != "empty"]
        if len(hs) >= 2:
            a, b = hs[0], hs[1]
            break
    else:
        raise AssertionError("no txn touches two accounts with storage")
    storage[b] = storage[a]
    state = _with_storage_root(state, b, acc[a][2])
    return blk, state, storage


def _one_of_two_in_map(oracle, seed):
    """Two accounts with the same storage root, only the first in the map; a txn reads a slot of the second."""
    blk, state, storage = _shared_tries(oracle, seed)
    blk.txns = copy.deepcopy(blk.txns)
    a, b = [h for h in storage if sum(1 for x in storage.values() if x is storage[h]) > 1][:2]
    del storage[b]
    # a txn reads a slot of the second
    for t in blk.txns:
        for addr, tr in t["traces"]:
            if oracle.keccak256(addr) == b:
                tr["storage_read"] = list(tr.get("storage_read") or []) + [bytes([0x11] * 32)]
                break
        else:
            continue
        break
    return blk, state, storage


def _bare_hash_and_empty_entries(oracle, seed, empty_root_hash):
    """A map entry that is a bare hash node (an account no txn reads the slots of) and an empty trie for an account with
    an empty root, next to other empty-rooted accounts outside the map; txns write slots of the empty entry and of an
    empty-rooted account outside the map.  empty_root_hash: one more empty-rooted account whose entry is a hash node of
    the empty root, first in key order (so the empty trie is still the empty-rooted trie witnessed last)."""
    blk = synth.gen_block(seed, n_accounts=80, n_txns=5, inline_code_frac=0.0, contract_frac=0.4, slots_lo=2, slots_hi=20)
    blk.txns = copy.deepcopy(blk.txns)
    state, storage = _direct(oracle, blk.flat)
    acc = _accounts(state)
    accessed = _accessed(oracle, blk)
    touched = _touched(oracle, blk)
    bare = [h for h in storage if h not in accessed and storage[h][0] != "empty"]
    assert bare
    storage[bare[0]] = ("hash", acc[bare[0]][2])
    empties = sorted(h for h in touched if h in acc and acc[h][2] == EMPTY_TRIE and h not in storage)
    assert len(empties) >= 4, len(empties)
    if empty_root_hash:
        storage[empties[0]] = ("hash", EMPTY_TRIE)
    storage[empties[1]] = ("empty",)
    for h in empties[1:3]:
        ti = min(touched[h])
        for addr, tr in blk.txns[ti]["traces"]:
            if oracle.keccak256(addr) == h:
                tr["storage_written"] = list(tr.get("storage_written") or []) + [(bytes([0x22] * 31 + [h[0]]), 5)]
                break
    return blk, state, storage


def _withheld(oracle, seed, step):
    """every storage trie withheld (step 1), or every other one (step 2)"""
    blk = synth.gen_block(seed, n_accounts=100, n_txns=4, inline_code_frac=0.0)
    state, storage = _direct(oracle, blk.flat)
    keep = {} if step == 1 else dict(sorted(storage.items())[::2])
    return blk, state, keep


# The product's host path and the oracle decode this input differently, a difference older than the device loop's
# by-address join.  The device loop is held to the host path here (test_default_equals_host_txn_path), as everywhere.
HOST_PATH_ONLY = {"empty_root_hash_entry"}


def _success_cases(oracle, lib):
    """(name, kind-2 FlatBlock, Combined FlatBlock of the same tries or None where the by-root join means something else)"""
    cases = []
    shapes = [
        ("c1", synth.gen_block(11, n_accounts=300, n_txns=6, inline_code_frac=0.0)),
        ("withdrawals", synth.gen_block(12, n_accounts=120, n_txns=3, n_withdrawals=2, inline_code_frac=0.0)),
        ("one_txn_dummy", synth.gen_block(13, n_accounts=80, n_txns=1, inline_code_frac=0.0)),
        ("no_txn", synth.gen_block(14, n_accounts=40, n_txns=0, n_withdrawals=1, inline_code_frac=0.0)),
    ]
    for name, blk in shapes:
        state, storage = _direct(oracle, blk.flat)
        cases.append((name, _kind2(blk.flat, state, storage), blk.flat))
    rng = np.random.default_rng(3)
    for i in range(4):
        blk = synth.gen_block(930 + i, n_accounts=40, n_txns=int(rng.integers(2, 8)), inline_code_frac=0.0, contract_frac=0.7, slots_lo=4, slots_hi=60,
                              slot_reads=(0, 4), slot_writes=(0, 6), zero_write_frac=0.6, accounts_per_txn=(2, 6))
        comb = _combined(lib, blk.flat, *_witness_like(oracle, blk, rng))
        # (back to direct nodes through the oracle: the accounts' storage-root fields then match the pruned tries)
        cases.append((f"witness_like_{i}", _kind2(blk.flat, *_direct(oracle, comb)), comb))
    blk, state, storage = _shared_tries(oracle, 940)
    cases.append(("shared_tries", _kind2(blk.flat, state, storage), _combined(lib, blk.flat, state, storage)))
    blk, state, storage = _one_of_two_in_map(oracle, 940)
    cases.append(("one_of_two_in_map", _kind2(blk.flat, state, storage), None))
    blk, state, storage = _bare_hash_and_empty_entries(oracle, 941, False)
    cases.append(("bare_hash_and_empty_entries", _kind2(blk.flat, state, storage), None))
    blk, state, storage = _bare_hash_and_empty_entries(oracle, 941, True)
    cases.append(("empty_root_hash_entry", _kind2(blk.flat, state, storage), None))
    for step in (1, 2):
        blk, state, storage = _withheld(oracle, 942, step)
        cases.append((f"withheld_{'all' if step == 1 else 'every_other'}", _kind2(blk.flat, state, storage), None))
    return cases


def _error_cases(oracle, lib):
    """Blocks the reference fails on (decoding.rs:31-49), as direct pre-images: (name, code, kind-2 FlatBlock)"""
    cases = []

    def base(**kw):
        return synth.gen_block(55, n_accounts=80, n_txns=3, n_withdrawals=1, inline_code_frac=0.0, **kw)

    def as_kind2(b):
        state, storage = _direct(oracle, b.flat)
        return _kind2(b.flat, state, storage)

    b = base()
    b.withdrawals = [(bytes(range(20)), 5)]
    cases.append(("withdrawal_to_missing_account", 25, as_kind2(b)))
    b = base(virtual_depth=3, virtual_accounts_log16=3)
    b.txns = copy.deepcopy(b.txns)
    b.txns[0]["traces"].append((bytes([7] * 20), {"balance": 1}))
    cases.append(("touched_account_behind_hash_node", 24, as_kind2(b)))
    b = synth.gen_block(55, n_accounts=80, n_txns=3, n_withdrawals=1, inline_code_frac=0.0, contract_frac=0.5, slots_hi=40)
    state, storage = _direct(oracle, b.flat)
    addr, tr = next((a, t) for a, t in b.txns[1]["traces"] if t.get("storage_read"))
    haddr, hslot = oracle.keccak256(addr), oracle.keccak256(tr["storage_read"][0])
    root = storage[haddr]
    if root[0] == "branch":
        ch = list(root[1])
        ch[hslot[0] >> 4] = ("hash", bytes([0x5A]) * 32)
        storage[haddr] = ("branch", ch, root[2])
    else:
        storage[haddr] = ("hash", bytes([0x5A]) * 32)
    cases.append(("storage_slot_behind_hash_node", 24, _kind2(b.flat, state, storage)))
    short = next(a for a in (i.to_bytes(20, "big") for i in range(1, 100000)) if oracle.keccak256(a)[0] == 0)
    b = base()
    b.txns = copy.deepcopy(b.txns)
    b.txns[1]["traces"].append((short, {"balance": 1}))
    cases.append(("hashed_address_with_a_leading_zero_byte", 42, as_kind2(b)))
    b = base(virtual_depth=3, virtual_accounts_log16=3)
    b.txns = copy.deepcopy(b.txns)
    b.txns[0]["traces"].append((bytes([7] * 20), {"balance": 1}))
    b.txns[2]["new_receipt_trie_node_byte"] = b"\xc1\x80"
    cases.append(("loop_error_in_txn_0_and_bad_receipt_in_txn_2", 43, as_kind2(b)))
    b = base(virtual_depth=3, virtual_accounts_log16=3)
    b.txns = copy.deepcopy(b.txns)
    b.txns[0]["traces"].append((bytes([7] * 20), {"balance": 1}))
    addr, tr = b.txns[1]["traces"][0]
    tr = dict(tr)
    tr.pop("code_write", None)
    tr["code_read"] = bytes([0xAB] * 32)
    b.txns[1]["traces"][0] = (addr, tr)
    cases.append(("loop_error_in_txn_0_and_unresolvable_code_in_txn_1", 61, as_kind2(b)))
    # one to three faults of different kinds at random txns
    rng = np.random.default_rng(6)
    kinds = ["behind_hash", "bad_receipt", "unresolvable_code", "short_haddr", "missing_withdrawal"]
    for case in range(10):
        n_txns = int(rng.integers(2, 6))
        b = synth.gen_block(760 + case, n_accounts=60, n_txns=n_txns, n_withdrawals=1, virtual_depth=3, virtual_accounts_log16=3, allow_new_accounts=False,
                            inline_code_frac=0.0)
        b.txns = copy.deepcopy(b.txns)
        for k in rng.choice(kinds, size=int(rng.integers(1, 4)), replace=False):
            t = int(rng.integers(0, n_txns))
            if k == "behind_hash":
                b.txns[t]["traces"].append((bytes([7] * 20), {"balance": 1}))
            elif k == "bad_receipt":
                b.txns[t]["new_receipt_trie_node_byte"] = b"\xc1\x80"
            elif k == "unresolvable_code":
                b.txns[t]["traces"].append((bytes([9] * 19 + [t]), {"code_read": bytes([0xAB] * 32)}))
            elif k == "short_haddr":
                b.txns[t]["traces"].append((short, {"balance": 1}))
            else:
                b.withdrawals = [(bytes(range(20)), 5)]
        cases.append((f"faults_{case}", None, as_kind2(b)))
    return cases


@pytest.fixture(scope="module")
def lib():
    from proof_protocol_decoder_b200.lib import load_library

    return load_library()


@pytest.fixture(scope="module")
def success_cases(oracle, lib):
    return _success_cases(oracle, lib)


@pytest.fixture(scope="module")
def error_cases(oracle, lib):
    return _error_cases(oracle, lib)


# ---------------------------------------------------------------------------------------------- CPU
@pytest.fixture(scope="module")
def directcheck():
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc is needed to build the check harness")
    res = subprocess.run(["make", "-C", CSRC, "directcheck"], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    return os.path.join(CSRC, "build", "directcheck")


def _harness(binary, tmp_path, flats):
    paths = []
    for i, f in enumerate(flats):
        p = tmp_path / f"d{i}.flat"
        p.write_bytes(f)
        paths.append(str(p))
    res = subprocess.run([binary] + paths, capture_output=True, text=True)
    return res, [ln for ln in res.stdout.splitlines() if ln.strip()]


def test_cases_are_what_they_claim(oracle, success_cases):
    """The special cases hold what their names say, and the oracle decodes every one of them."""
    by = {n: (k2, comb) for n, k2, comb in success_cases}
    for name, k2, comb in success_cases:
        want = oracle.block_decode(k2)
        if comb is not None:
            assert oracle.block_decode(comb) == want, name
    state, storage = flat.parse_direct_pre_image(flat.pre_image_of(by["shared_tries"][0])[1])
    acc = _accounts(state)
    same = [h for h in storage if sum(1 for x in storage.values() if x == storage[h]) > 1 and storage[h][0] == "branch"]
    assert len(same) >= 2 and acc[same[0]][2] == acc[same[1]][2]
    state, storage = flat.parse_direct_pre_image(flat.pre_image_of(by["bare_hash_and_empty_entries"][0])[1])
    kinds = [t[0] for t in storage.values()]
    assert "hash" in kinds and "empty" in kinds and ("hash", EMPTY_TRIE) not in list(storage.values())
    state, storage = flat.parse_direct_pre_image(flat.pre_image_of(by["empty_root_hash_entry"][0])[1])
    assert ("hash", EMPTY_TRIE) in list(storage.values())
    state, storage = flat.parse_direct_pre_image(flat.pre_image_of(by["withheld_all"][0])[1])
    assert storage == {}


def test_device_loop_and_by_address_join_match_the_host_path(directcheck, tmp_path, success_cases):
    """Every success case: the join's arrays equal the host path's storage map account by account, and the device loop
    builds the same tries as the host loop, txn by txn."""
    res, lines = _harness(directcheck, tmp_path, [k2 for _, k2, _ in success_cases])
    assert res.returncode == 0 and len(lines) == len(success_cases), "\n".join(lines[-20:]) + res.stderr[-2000:]
    for (name, _, _), ln in zip(success_cases, lines):
        assert ln.endswith("identical"), (name, ln)


def test_device_side_hands_over_every_block_the_host_path_fails(directcheck, tmp_path, oracle, error_cases):
    from ppd_oracle_lib import OracleError

    res, lines = _harness(directcheck, tmp_path, [f for _, _, f in error_cases])
    assert len(lines) == len(error_cases), res.stdout[-2000:] + res.stderr[-2000:]
    seen = set()
    for (name, code, f), ln in zip(error_cases, lines):
        with pytest.raises(OracleError) as eo:
            oracle.block_decode(f)
        if code is not None:
            assert eo.value.code == code, name
        m = re.search(r": status (\d+) \((.*)\) from the host path; the device path (declines|raises flag)", ln)
        assert m, (name, ln)
        assert (int(m.group(1)), m.group(2)) == (eo.value.code, eo.value.msg), (name, ln)
        seen.add(eo.value.code)
    assert len(seen) >= 4, seen


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    from proof_protocol_decoder_b200.lib import Context, PpdError

    try:
        c = Context(0)
    except PpdError as e:
        pytest.skip(f"no usable CUDA device: {e}")
    yield c
    c.close()


@pytest.mark.gpu
def test_product_equals_oracle_on_the_device_loop(ctx, oracle, success_cases):
    for name, k2, comb in success_cases:
        want = oracle.block_decode(k2)
        got = ctx.block_decode(k2)
        st = ctx.stats()
        if name not in HOST_PATH_ONLY:
            assert got == want, name
        assert st["txn_loops_on_gpu"] == 1, name
        if comb is not None:
            assert oracle.block_decode(comb) == want, name
    # the contrast: the Combined form of the shared tries is joined by root, shares one expanded trie between two
    # accounts, and the device hands the block to the host path
    comb = next(c for n, _, c in success_cases if n == "shared_tries")
    assert ctx.block_decode(comb) == oracle.block_decode(comb)
    assert ctx.stats()["txn_loops_on_gpu"] == 0


@pytest.mark.gpu
def test_default_equals_host_txn_path(ctx, success_cases, monkeypatch):
    dev = [ctx.block_decode(k2) for _, k2, _ in success_cases]
    monkeypatch.setenv("PPD_HOST_TXN", "1")
    for (name, k2, _), d in zip(success_cases, dev):
        assert ctx.block_decode(k2) == d, name
        assert ctx.stats()["txn_loops_on_gpu"] == 0


@pytest.mark.gpu
def test_error_blocks_report_what_the_host_path_reports(ctx, oracle, error_cases, monkeypatch):
    from ppd_oracle_lib import OracleError
    from proof_protocol_decoder_b200.lib import PpdError

    def run(f):
        with pytest.raises(PpdError) as e:
            ctx.block_decode(f)
        return e.value.code, ctx.lib.L.ppd_last_error(ctx.h).decode(), ctx.stats()["txn_loops_on_gpu"]

    got = [run(f) for _, _, f in error_cases]
    monkeypatch.setenv("PPD_HOST_TXN", "1")
    for (name, _, f), g in zip(error_cases, got):
        with pytest.raises(OracleError) as eo:
            oracle.block_decode(f)
        h = run(f)
        assert g[0] == h[0] == eo.value.code, name
        assert g[1] == h[1], name
        assert g[2] == 0, name


@pytest.mark.gpu
def test_payload_crosses_pcie_once(ctx, lib, success_cases):
    k2 = success_cases[0][1]
    wit = lib.direct_to_compact(flat.pre_image_of(k2)[1])
    ctx.block_decode(k2)
    st = ctx.stats()
    assert st["txn_loops_on_gpu"] == 1
    assert st["h2d_bytes"] < len(k2) + len(wit)


@pytest.mark.gpu
def test_full_size_config_2_block(ctx, oracle, monkeypatch):
    monkeypatch.delenv("PPD_GPU_PARSE_MIN_BYTES", raising=False)  # the production threshold: a C2 witness clears it
    monkeypatch.delenv("PPD_GPU_DUMP_MIN_TOUCHED", raising=False)
    blk = synth.gen_block(
        2, n_accounts=20000, n_txns=200, contract_frac=0.15, slots_lo=1, slots_hi=4096, virtual_depth=7, accounts_per_txn=(80, 120), slot_reads=(0, 3),
        slot_writes=(0, 3), allow_new_accounts=False, allow_self_destruct=False, inline_code_frac=0.0,
    )
    state, storage = _direct(oracle, blk.flat)
    k2 = _kind2(blk.flat, state, storage)
    got = ctx.block_decode(k2)
    assert ctx.stats()["txn_loops_on_gpu"] == 1
    assert got == oracle.block_decode(k2) == oracle.block_decode(blk.flat)


def _mixed(success_cases, n):
    """n FlatBlocks, kind 0 and kind 2 mixed so that a lane (block i runs on lane i mod 64) meets both joins"""
    pairs = [(k2, comb) for _, k2, comb in success_cases if comb is not None]
    out = []
    for i in range(n):
        k2, comb = pairs[i % len(pairs)]
        out.append(k2 if (i + i // 64) % 2 == 0 else comb)
    return out


@pytest.mark.gpu
def test_batch_and_stream_mix_kinds_across_lanes_and_replay(ctx, success_cases):
    flats = _mixed(success_cases, 150)
    single = {f: ctx.block_decode(f) for f in set(flats)}
    outs = ctx.blocks_decode_batch(flats)
    assert ctx.stats()["txn_loops_on_gpu"] >= sum(1 for f in flats if flat.pre_image_of(f)[0] == flat.PRE_IMAGE_DIRECT)
    for f, o in zip(flats, outs):
        assert o == single[f]
    ms = ctx.replay_last(ctx.REPLAY_ALL)
    assert ms >= 0
    assert ctx.blocks_decode_batch(flats) == outs
    got = [None] * len(flats)

    def done(i, r):
        with r:
            got[i] = bytes(r.view)

    ctx.blocks_decode_stream(flats, done)
    assert got == outs
    ctx.replay_last(ctx.REPLAY_ALL)
    assert ctx.blocks_decode_batch(flats) == outs
