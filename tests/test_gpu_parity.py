"""Parity of the CUDA path (through the C ABI) with the CPU oracle and the reference goldens.
Run on the B200 box: python -m pytest tests -m gpu"""
import numpy as np
import pytest

from ppd_oracle_lib import OracleError, parse_pre_image_dump

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from proof_protocol_decoder_b200.lib import Context

    c = Context(0)
    yield c
    c.close()


def _batch(msgs):
    data = np.frombuffer(b"".join(msgs), dtype=np.uint8) if msgs else np.zeros(0, np.uint8)
    off = np.zeros(len(msgs) + 1, dtype=np.uint64)
    np.cumsum([len(m) for m in msgs], out=off[1:])
    return data, off


def test_keccak_batch_edges(ctx, oracle, goldens):
    rng = np.random.default_rng(0)
    lens = [0, 1, 20, 32, 55, 56, 134, 135, 136, 137, 271, 272, 273, 407, 408, 409, 1000, 4096]
    msgs = [rng.bytes(n) for n in lens] + [b"\x80"]
    data, off = _batch(msgs)
    got = ctx.keccak256_batch(data, off)
    want = oracle.keccak256_batch(data, off)
    assert (got == want).all()
    assert got[0].tobytes().hex() == goldens["constants"]["EMPTY_CODE_HASH"]
    assert got[-1].tobytes().hex() == goldens["constants"]["EMPTY_TRIE_HASH"]


def test_keccak_batch_random_lengths(ctx, oracle):
    rng = np.random.default_rng(1)
    lens = rng.integers(0, 4097, size=3000)
    msgs = [rng.bytes(int(n)) for n in lens]
    data, off = _batch(msgs)
    assert (ctx.keccak256_batch(data, off) == oracle.keccak256_batch(data, off)).all()


def test_keccak_batch_addresses_and_slots(ctx, oracle):
    rng = np.random.default_rng(2)
    for width in (20, 32):
        n = 100_000
        data = np.frombuffer(rng.bytes(width * n), dtype=np.uint8)
        off = (np.arange(n + 1, dtype=np.uint64) * width).astype(np.uint64)
        assert (ctx.keccak256_batch(data, off) == oracle.keccak256_batch(data, off)).all()


@pytest.mark.parametrize("idx", range(6))
def test_golden_state_roots_on_gpu(ctx, oracle, goldens, idx):
    from proof_protocol_decoder_b200 import flat

    g = goldens["compact_goldens"][idx]
    w = bytes.fromhex(g["witness_hex"])
    d = flat.parse_pre_image_dump(ctx.compact_decode(w))
    assert d["version"] == 1
    assert d["state_root"].hex() == g["state_root"]
    o = parse_pre_image_dump(oracle.compact_decode(w))
    assert d["storage"] == o["storage"]
    assert d["code"] == o["code"]


def test_header_only_and_simple_payload(ctx, oracle, goldens):
    from proof_protocol_decoder_b200 import flat

    d = flat.parse_pre_image_dump(ctx.compact_decode(b"\x01"))
    assert d["state_root"].hex() == goldens["constants"]["EMPTY_TRIE_HASH"]


@pytest.mark.parametrize(
    "witness",
    [b"", b"\x01\x07", b"\x01\x05\x41\x10", b"\x01\x00\x58", b"\x01\x03\x00", b"\x01\x06\x06", b"\x01\x06\x02\x03", b"\x01\x06\x02\x1a\x00\x01\x00\x00"],
)
def test_compact_error_variants_match_oracle(ctx, oracle, witness):
    from proof_protocol_decoder_b200 import PpdError

    with pytest.raises(OracleError) as eo:
        oracle.compact_decode(witness)
    with pytest.raises(PpdError) as eg:
        ctx.compact_decode(witness)
    assert eg.value.code == eo.value.code


def test_blocks_stream_hands_every_block_over_once(ctx, oracle):
    """ppd_blocks_decode_stream: the same bytes as ppd_blocks_decode_batch, each block delivered exactly once through the
    callback (in completion order), a failing block with its status."""
    from proof_protocol_decoder_b200 import PpdError, synth

    blocks = [synth.gen_block(300 + i, n_accounts=60 + 10 * i, n_txns=3 + i % 3, n_withdrawals=i % 2) for i in range(9)]
    bad = synth.gen_block(3, n_accounts=50, n_txns=1)
    bad.withdrawals = [(b"\x11" * 20, 5)]  # not in the state trie: MissingWithdrawalAccount
    flats = [b.flat for b in blocks] + [bad.flat]
    got = {}

    def on_done(i, o):
        assert i not in got
        if isinstance(o, Exception):
            got[i] = o
        else:
            got[i] = bytes(o.view)
            o.close()

    ctx.blocks_decode_stream(flats, on_done)
    assert sorted(got) == list(range(len(flats)))
    for i, b in enumerate(blocks):
        assert got[i] == oracle.block_decode(b.flat)
    assert isinstance(got[len(blocks)], PpdError) and got[len(blocks)].code == 25


def test_balance_wider_than_256_bits_is_the_u256_panic(ctx, oracle):
    """read_cbor_u256 reads the byte vector and U256::from_big_endian panics on more than 32 bytes
    (compact_prestate_processing.rs): a panic site (status 47), not CompactParsingError::InvalidByteVector."""
    import witness_shapes as ws
    from proof_protocol_decoder_b200 import PpdError

    wide = ws.HDR + ws.account(ws.nibs("a" * 63), balance=1 << 263) + ws.account(ws.nibs("b" * 63), balance=9) + ws.branch((1 << 10) | (1 << 11))
    with pytest.raises(OracleError) as eo:
        oracle.compact_decode(wide)
    with pytest.raises(PpdError) as eg:
        ctx.compact_decode(wide)
    assert eo.value.code == eg.value.code == 47


def _check_block(ctx, oracle, blk):
    f = blk.flat
    want = oracle.block_decode(f)
    got = ctx.block_decode(f)
    if got != want:
        from proof_protocol_decoder_b200 import flat

        a, b = flat.parse_ir_dump(got), flat.parse_ir_dump(want)
        assert len(a) == len(b)
        for i, (x, y) in enumerate(zip(a, b)):
            for k in x:
                assert x[k] == y[k], f"IR {i} field {k} differs"
    assert got == want
    return got


@pytest.mark.parametrize("seed", [1, 2, 3, 4, 5])
def test_c1_blocks_bit_exact(ctx, oracle, seed):
    from proof_protocol_decoder_b200 import synth

    _check_block(ctx, oracle, synth.gen_block(seed, n_accounts=1000, n_txns=10, n_withdrawals=seed % 3))


@pytest.mark.parametrize("n_txns,n_wd", [(0, 0), (0, 2), (1, 0), (1, 2), (2, 0), (2, 3)])
def test_dummy_padding_and_withdrawals_unpinned(ctx, oracle, n_txns, n_wd):
    """(unpinned: the dummy entries' subset key 0_u64 as zero nibbles is this repo's reading of eth_trie_utils, shared by the
    oracle; no reference fixture covers it — DESIGN.md section 8)"""
    from proof_protocol_decoder_b200 import synth

    _check_block(ctx, oracle, synth.gen_block(100 + n_txns * 10 + n_wd, n_accounts=120, n_txns=n_txns, n_withdrawals=n_wd))


def test_tiny_states(ctx, oracle):
    from proof_protocol_decoder_b200 import synth

    for n in (0, 1, 2, 3):
        _check_block(ctx, oracle, synth.gen_block(200 + n, n_accounts=n, n_txns=2, allow_self_destruct=False))


def test_mainnet_shaped_block_scaled(ctx, oracle):
    from proof_protocol_decoder_b200 import synth

    blk = synth.gen_block(
        2, n_accounts=2000, n_txns=20, contract_frac=0.15, slots_hi=512, virtual_depth=5, virtual_accounts_log16=5,
        accounts_per_txn=(40, 60), slot_reads=(0, 3), slot_writes=(0, 3), allow_new_accounts=False, allow_self_destruct=False,
    )
    _check_block(ctx, oracle, blk)


def test_blocks_batch_matches_single(ctx, oracle):
    from proof_protocol_decoder_b200 import synth

    blks = [synth.gen_block(300 + i, n_accounts=150, n_txns=3, n_withdrawals=i % 2) for i in range(6)]
    outs = ctx.blocks_decode_batch([b.flat for b in blks])
    for b, o in zip(blks, outs):
        assert o == oracle.block_decode(b.flat)


def test_reference_interface_mirror(ctx, oracle):
    from proof_protocol_decoder_b200 import flat, synth

    blk = synth.gen_block(11, n_accounts=100, n_txns=3, n_withdrawals=1)
    bt, meta, other = blk.to_block_trace()
    irs = bt.into_txn_proof_gen_ir(meta, other, ctx=ctx)
    want = flat.parse_ir_dump(oracle.block_decode(bt.to_flat(meta, other)))
    assert irs == want
    assert len(irs) == 4  # 3 txns + the withdrawal dummy (decoding.rs:367-387)
    assert irs[-1]["withdrawals"] and irs[-1]["signed_txn"] is None


@pytest.mark.parametrize("n", [0, 1, 2, 3, 17, 1000, 50_000])
def test_sorted_leaves_root(ctx, oracle, n):
    from proof_protocol_decoder_b200 import synth

    keys, val_off, vals = synth.gen_sorted_leaves(n, seed=n + 1)
    assert ctx.trie_root_sorted_leaves(keys, val_off, vals) == oracle.trie_root_from_leaves(keys, val_off, vals)


def test_sorted_leaves_shared_prefixes_and_small_values(ctx, oracle):
    # long shared prefixes force extension nodes; tiny values force nodes shorter than 32 bytes (inlined refs)
    rng = np.random.default_rng(3)
    n = 4000
    keys = np.zeros((n, 32), dtype=np.uint8)
    keys[:, :28] = np.frombuffer(rng.bytes(28), dtype=np.uint8)
    keys[:, 28:] = np.frombuffer(rng.bytes(4 * n), dtype=np.uint8).reshape(n, 4)
    keys[: n // 2, 5] ^= 0x10
    keys = np.unique(keys, axis=0)
    be = keys.view(">u8")
    keys = np.ascontiguousarray(keys[np.lexsort((be[:, 3], be[:, 2], be[:, 1], be[:, 0]))])
    n = len(keys)
    lens = rng.integers(1, 4, size=n).astype(np.uint64)
    val_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=val_off[1:])
    vals = np.frombuffer(rng.bytes(int(val_off[-1])), dtype=np.uint8)
    assert ctx.trie_root_sorted_leaves(keys, val_off, vals) == oracle.trie_root_from_leaves(keys, val_off, vals)


def test_unsorted_keys_are_rejected(ctx):
    from proof_protocol_decoder_b200 import PpdError, synth

    keys, val_off, vals = synth.gen_sorted_leaves(100, seed=9)
    duplicated = keys.copy()
    duplicated[51] = duplicated[50]  # still ascending, but one key twice
    for bad in (keys[::-1].copy(), duplicated):
        with pytest.raises(PpdError) as e:
            ctx.trie_root_sorted_leaves(bad, val_off, vals)
        assert e.value.code == 63


def test_sorted_leaves_root_one_million(ctx, oracle):
    # config 5 at 1 % of its full size: the largest the CPU oracle finishes in seconds
    from proof_protocol_decoder_b200 import synth

    keys, val_off, vals = synth.gen_sorted_leaves(1_000_000, seed=5)
    assert ctx.trie_root_sorted_leaves(keys, val_off, vals) == oracle.trie_root_from_leaves(keys, val_off, vals)


def test_sorted_leaves_root_independent_of_value_alignment(ctx):
    # size-independent property usable at full scale: the root of N leaves does not change when the
    # value pool is shifted by 1..3 bytes (every value at a different alignment), and does change
    # when one bit of one value changes
    from proof_protocol_decoder_b200 import synth

    keys, val_off, vals = synth.gen_sorted_leaves(300_000, seed=8)
    r0 = ctx.trie_root_sorted_leaves(keys, val_off, vals)
    for k in (1, 2, 3):
        shifted = np.concatenate([np.full(k, 0xEE, np.uint8), vals])
        assert ctx.trie_root_sorted_leaves(keys, val_off + np.uint64(k), shifted) == r0
    vals2 = vals.copy()
    vals2[int(val_off[123456])] ^= 1
    assert ctx.trie_root_sorted_leaves(keys, val_off, vals2) != r0


def test_storage_heavy_tries_sharded(ctx, oracle):
    # config 3 in miniature through the sharding layer (world size 1 here; two ranks: test_sharding_gloo.py)
    from proof_protocol_decoder_b200 import shard, synth

    sizes = [50_000, 50_000, 20_000, 7, 1]
    tries = [synth.gen_sorted_leaves(n, seed=70 + i, val_lo=1, val_hi=33) for i, n in enumerate(sizes)]
    got = shard.sharded_trie_roots(lambda i: ctx.trie_root_sorted_leaves(*tries[i]), sizes)
    assert got == [oracle.trie_root_from_leaves(*t) for t in tries]


def test_batch_larger_than_lane_count_with_a_bad_block(ctx, oracle):
    from proof_protocol_decoder_b200 import PpdError, synth

    blks = [synth.gen_block(400 + i, n_accounts=80 + 5 * i, n_txns=i % 4, n_withdrawals=i % 3) for i in range(24)]
    flats = [b.flat for b in blks]
    bad = bytearray(flats[7])
    # corrupt the compact header version (first byte of the witness, after magic/version/kind/len)
    bad[16] = 2
    flats[7] = bytes(bad)
    outs = ctx.blocks_decode_batch(flats)
    for i, (f, o) in enumerate(zip(flats, outs)):
        if i == 7:
            assert isinstance(o, PpdError) and o.code == 40
        else:
            assert o == oracle.block_decode(f), f"block {i}"


def _mutations(w: bytes, rng, n):
    out = []
    for _ in range(n):
        b = bytearray(w)
        kind = rng.integers(0, 6)
        if kind == 0 and len(b) > 2:  # flip one byte
            i = int(rng.integers(1, len(b)))
            b[i] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1 and len(b) > 2:  # truncate
            b = b[: int(rng.integers(1, len(b)))]
        elif kind == 2:  # insert a random byte
            i = int(rng.integers(1, len(b) + 1))
            b[i:i] = bytes([int(rng.integers(0, 256))])
        elif kind == 3 and len(b) > 4:  # delete a short slice
            i = int(rng.integers(1, len(b) - 1))
            del b[i : i + int(rng.integers(1, 4))]
        elif kind == 4 and len(b) > 8:  # duplicate a slice
            i = int(rng.integers(1, len(b) - 4))
            k = int(rng.integers(1, 40))
            b[i:i] = b[i : i + k]
        else:  # overwrite an opcode-looking byte
            i = int(rng.integers(1, len(b)))
            b[i] = int(rng.integers(0, 8))
        out.append(bytes(b))
    return out


def test_mutated_witnesses_same_status_or_same_result(ctx, oracle, goldens):
    # robustness parity (SURVEY 8f-4): corrupt witnesses must fail with the same status as the oracle,
    # and the ones that still decode must decode to the same tries
    from proof_protocol_decoder_b200 import PpdError, flat, synth

    rng = np.random.default_rng(2024)
    seeds = [bytes.fromhex(g["witness_hex"]) for g in goldens["compact_goldens"]]
    blk = synth.gen_block(31, n_accounts=40, n_txns=1, virtual_depth=3, virtual_accounts_log16=3, contract_frac=0.3)
    bt, _, _ = blk.to_block_trace()
    seeds.append(bytes(bt.trie_pre_images["combined"]["compact"]))
    n_err = n_ok = 0
    for w in seeds:
        for m in _mutations(w, rng, 120):
            try:
                want = parse_pre_image_dump(oracle.compact_decode(m))
                want_code = 0
            except OracleError as e:
                want, want_code = None, e.code
            try:
                got = flat.parse_pre_image_dump(ctx.compact_decode(m))
                got_code = 0
            except PpdError as e:
                got, got_code = None, e.code
            assert got_code == want_code, f"status {got_code} vs oracle {want_code} for witness {m.hex()}"
            if want is not None:
                assert got["state_root"] == want["state_root"] and got["storage"] == want["storage"] and got["code"] == want["code"], m.hex()
                n_ok += 1
            else:
                n_err += 1
    assert n_err > 100 and n_ok > 20


def _error_cases():
    """(name, FlatBlock) pairs that must fail: each is a valid synthetic block with one thing broken."""
    import copy
    import struct

    from proof_protocol_decoder_b200 import synth

    def base(**kw):
        return synth.gen_block(55, n_accounts=80, n_txns=3, n_withdrawals=1, **kw)

    cases = []
    b = base()
    b.withdrawals = [(bytes(range(20)), 5)]  # an account that is not in the state trie
    cases.append(("withdrawal_to_missing_account", b.flat))

    b = base(virtual_depth=3, virtual_accounts_log16=3)
    b.txns = copy.deepcopy(b.txns)
    b.txns[0]["traces"].append((bytes([7] * 20), {"balance": 1}))  # its path runs into a hashed-out subtree
    cases.append(("touched_account_behind_hash_node", b.flat))

    b = base()
    b.txns = copy.deepcopy(b.txns)
    addr, tr = b.txns[1]["traces"][0]
    tr = dict(tr)
    tr.pop("code_write", None)
    tr["code_read"] = bytes([0xAB] * 32)  # nobody can resolve this hash
    b.txns[1]["traces"][0] = (addr, tr)
    cases.append(("unresolvable_code_hash", b.flat))

    b = base()
    b.txns = copy.deepcopy(b.txns)
    b.txns[2]["new_receipt_trie_node_byte"] = b"\xc1\x80"  # a list that is not a legacy receipt
    cases.append(("receipt_neither_legacy_nor_string", b.flat))

    b = base()
    f = bytearray(b.flat)
    cases.append(("truncated_flat_block", bytes(f[: len(f) // 2])))
    f2 = bytearray(b.flat)
    struct.pack_into("<I", f2, 8, 1)  # pre_image_kind = Separate: todo!() in the reference
    cases.append(("unimplemented_pre_image_kind", bytes(f2)))

    b = base()
    b.compact = b"\x02" + b.compact[1:]  # header version 2: assert at processed_block_trace.rs:175
    cases.append(("incompatible_header_version", b.flat))
    return cases


@pytest.mark.parametrize("name,flat_block", _error_cases(), ids=[c[0] for c in _error_cases()])
def test_block_error_statuses_match_oracle(ctx, oracle, name, flat_block):
    from proof_protocol_decoder_b200 import PpdError

    with pytest.raises(OracleError) as eo:
        oracle.block_decode(flat_block)
    with pytest.raises(PpdError) as eg:
        ctx.block_decode(flat_block)
    assert eg.value.code == eo.value.code, f"{name}: {eg.value} vs {eo.value}"
    # the context stays usable after a failed block
    from proof_protocol_decoder_b200 import synth

    ok = synth.gen_block(56, n_accounts=30, n_txns=1).flat
    assert ctx.block_decode(ok) == oracle.block_decode(ok)


# ---- the witness parse / pre-image arena on the GPU (ppd_parse.cu) against the host builder --------------
def _both_builders(ctx, fn):
    """fn() with the GPU witness parser, then with the host one (PPD_HOST_PARSE); returns both results and stats."""
    import os

    os.environ.pop("PPD_HOST_PARSE", None)
    a = fn()
    sa = ctx.stats()
    os.environ["PPD_HOST_PARSE"] = "1"
    try:
        b = fn()
        sb = ctx.stats()
    finally:
        os.environ.pop("PPD_HOST_PARSE", None)
    return a, sa, b, sb


@pytest.mark.parametrize("idx", range(6))
def test_gpu_parse_goldens_match_host_builder(ctx, oracle, goldens, idx):
    g = goldens["compact_goldens"][idx]
    wit = bytes.fromhex(g["witness_hex"])
    a, sa, b, sb = _both_builders(ctx, lambda: ctx.compact_decode(wit))
    assert a == b
    assert parse_pre_image_dump(a)["state_root"].hex() == g["state_root"]
    assert sb["witnesses_on_gpu"] == 0
    # every golden is a canonical witness (SURVEY 7): the GPU builder must have taken all of them
    assert sa["witnesses_on_gpu"] == 1, "the GPU parser declined a canonical golden witness"
    assert sa["nodes_hashed"] == sb["nodes_hashed"] and sa["node_permutations"] == sb["node_permutations"]


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_gpu_parse_blocks_match_host_builder(ctx, oracle, seed):
    from proof_protocol_decoder_b200 import synth

    blk = synth.gen_block(40 + seed, n_accounts=1500, n_txns=8, contract_frac=0.2, slots_hi=256, virtual_depth=4,
                          virtual_accounts_log16=5, accounts_per_txn=(20, 40), slot_reads=(0, 3), slot_writes=(0, 3),
                          allow_new_accounts=False, allow_self_destruct=False)
    a, sa, b, sb = _both_builders(ctx, lambda: ctx.block_decode(blk.flat))
    assert a == b == oracle.block_decode(blk.flat)
    assert sa["witnesses_on_gpu"] == 1 and sb["witnesses_on_gpu"] == 0
    assert sa["witness_instructions"] > 1500
    # (with the witness parsed on the GPU the txn loop runs there too and builds fewer unobserved trie versions than the
    # host loop, which the host-parsed block takes: the node counts of the two differ, the outputs do not)
    assert sa["txn_loops_on_gpu"] == 1 and sb["txn_loops_on_gpu"] == 0
    assert sa["nodes_hashed"] <= sb["nodes_hashed"]


def test_gpu_parse_declines_non_canonical_and_malformed(ctx, oracle, goldens):
    """Witnesses the GPU builder must hand to the host builder: results and statuses still match the oracle."""
    import witness_shapes as ws

    cases = [p[1] for p in ws.PAIRS]
    for wit in cases:
        try:
            want = oracle.compact_decode(wit)
        except OracleError as e:
            with pytest.raises(Exception) as ei:
                ctx.compact_decode(wit)
            assert getattr(ei.value, "code", None) == e.code
            continue
        assert ctx.compact_decode(wit) == want
        assert ctx.stats()["witnesses_on_gpu"] == 0


@pytest.mark.parametrize("sizes", [
    [20000] * 8,                                  # every code string spans five tiles
    [3000, 40000, 17, 24000, 33000, 1, 9000, 45000, 12000],  # mixed: some longer than a whole tile group's first tile
    [70000, 70000],                               # longer than a tile group (8 tiles) of a small witness
])
def test_gpu_parse_long_code_strings_jump_tiles_and_groups(ctx, oracle, sizes):
    import witness_shapes as ws

    wit = ws.long_code_witness(sizes)
    want = oracle.compact_decode(wit)
    got = ctx.compact_decode(wit)
    st = ctx.stats()
    assert got == want
    assert st["witnesses_on_gpu"] == 1
    assert st["witness_instructions"] == 2 * len(sizes) + 1
    assert len(parse_pre_image_dump(got)["code"]) == len(sizes)  # one code map entry per (distinct, random) code string


def test_gpu_parse_size_threshold(ctx, oracle):
    """Production default: witnesses under 512 KiB take the host builder, larger ones the GPU parser; same bytes out."""
    import os

    import witness_shapes as ws

    small = ws.long_code_witness([20000] * 4)      # 80 KB
    big = ws.long_code_witness([60000] * 12)       # 720 KB
    saved = os.environ.pop("PPD_GPU_PARSE_MIN_BYTES", None)
    try:
        for wit, on_gpu in ((small, 0), (big, 1)):
            assert ctx.compact_decode(wit) == oracle.compact_decode(wit)
            assert ctx.stats()["witnesses_on_gpu"] == on_gpu
    finally:
        if saved is not None:
            os.environ["PPD_GPU_PARSE_MIN_BYTES"] = saved


@pytest.mark.parametrize("seed", range(12))
def test_gpu_parse_random_shapes_verified_against_host_builder(ctx, oracle, seed):
    """Random block shapes (hashed-out siblings at several depths, storage tries from one slot to hundreds, with and
    without contracts) decoded with PPD_VERIFY_GPU_PARSE: the library itself compares the GPU-built pre-image with the
    host builder's node by node (keys, values, hashes, account records, levels, per-account maps) and fails on any
    difference; the result must also equal the oracle's."""
    import os

    from proof_protocol_decoder_b200 import synth

    rng = np.random.default_rng(1000 + seed)
    vdepth = int(rng.integers(0, 6))
    blk = synth.gen_block(
        500 + seed, n_accounts=int(rng.integers(1, 900)), n_txns=int(rng.integers(0, 5)), contract_frac=float(rng.choice([0.0, 0.1, 0.5, 1.0])),
        slots_hi=int(rng.choice([1, 8, 300])), virtual_depth=vdepth, virtual_accounts_log16=max(vdepth, 4),
        accounts_per_txn=(1, 12), slot_reads=(0, 3), slot_writes=(0, 3), allow_new_accounts=vdepth == 0, allow_self_destruct=vdepth == 0,
    )
    os.environ["PPD_VERIFY_GPU_PARSE"] = "1"
    try:
        got = ctx.block_decode(blk.flat)
    finally:
        os.environ.pop("PPD_VERIFY_GPU_PARSE", None)
    assert ctx.stats()["witnesses_on_gpu"] == 1
    assert got == oracle.block_decode(blk.flat)


def test_full_size_config2_block_bit_exact(ctx, oracle):
    """BASELINE.json configs[1] at full size (20k touched accounts in a virtual 16^7-account state, 200 txns: a 36 MB
    witness, 1.05 M instructions, 52 MB of IR): the bench's own block, decoded with production thresholds (GPU witness
    parser, GPU IR dump), byte for byte against the CPU oracle."""
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench

    flat = bench.c2_block(2, 1.0)
    saved = {k: os.environ.pop(k, None) for k in ("PPD_GPU_PARSE_MIN_BYTES", "PPD_GPU_DUMP_MIN_TOUCHED")}
    try:
        got = ctx.block_decode(flat)
        st = ctx.stats()
    finally:
        for k, v in saved.items():
            if v is not None:
                os.environ[k] = v
    assert st["witnesses_on_gpu"] == 1 and st["witness_instructions"] > 1_000_000
    assert st["txn_loops_on_gpu"] == 1, "the bench's block fell back to the host path (a flag of the device txn loop or of the IR layout)"
    want = oracle.block_decode(flat)
    assert len(got) == len(want) > 50_000_000
    assert got == want


def test_gpu_parse_leaf_value_lengths(ctx, oracle):
    """rlp_str(value) of a storage leaf (compact_to_partial_trie.rs:119) as the GPU emitter writes it: the single byte
    below 0x80 that is its own encoding, short strings, and every width of the long-string header."""
    import witness_shapes as ws

    for n in (1, 2, 31, 32, 55, 56, 57, 255, 256, 257, 65535, 65536, 70001):
        for first in (0x05, 0x80):
            val = bytes([first]) + bytes((7 * i + n) & 255 for i in range(n - 1))
            storage = ws.leaf(ws.nibs("3" * 64), val)
            wit = ws.HDR + ws.account_with_storage(ws.nibs("a" * 63), storage) + ws.account(ws.nibs("b" * 63), balance=9) + ws.branch((1 << 10) | (1 << 11))
            want = oracle.compact_decode(wit)
            assert ctx.compact_decode(wit) == want, f"value of {n} bytes starting with {first:#x}"
            assert ctx.stats()["witnesses_on_gpu"] == 1


def test_gpu_parse_stream_lengths_around_tile_boundaries(ctx, oracle):
    """Witness lengths of exactly k tiles (4 KiB), one byte less and one byte more, and a last instruction that ends
    exactly on a tile boundary: the boundary search's end-of-stream handling."""
    import witness_shapes as ws

    def witness(code_len):
        body = bytes((i * 31 + 7) & 255 for i in range(code_len))
        return (ws.HDR + ws.account_with_code(ws.nibs("1" * 63), ws.code(body), code_len) + ws.account(ws.nibs("2" * 63), balance=3)
                + ws.branch((1 << 1) | (1 << 2)))

    base = len(witness(1000)) - 1000
    seen = set()
    for tiles in (1, 2, 3, 8, 9, 16):
        for delta in (-2, -1, 0, 1, 2):
            target = tiles * 4096 + delta
            code_len = target - base
            wit = witness(code_len)
            for fix in range(4):  # the CBOR heads grow with the length: step until the total matches
                if len(wit) == target:
                    break
                code_len += target - len(wit)
                wit = witness(code_len)
            seen.add(len(wit) % 4096)
            assert ctx.compact_decode(wit) == oracle.compact_decode(wit), f"witness of {len(wit)} bytes"
            assert ctx.stats()["witnesses_on_gpu"] == 1
    assert {0, 1, 2, 4094, 4095} <= seen


def test_subset_marking_on_the_device_and_error_order(ctx, oracle):
    """create_trie_subset's marking walks (decoding.rs:185-209) are the walks of the device txn loop (txn_core.h:
    batch_walk).  A txn that touches a key under a hashed-out node is MissingKeysCreatingSubPartialTrie in the reference,
    possibly after other errors of earlier txns: the device loop only flags it, the host path then redoes the block
    and reports errors in the reference's order."""
    from proof_protocol_decoder_b200 import synth

    blk = synth.gen_block(77, n_accounts=1200, n_txns=12, contract_frac=0.3, slots_hi=64, virtual_depth=3, virtual_accounts_log16=5,
                          accounts_per_txn=(20, 40), slot_reads=(0, 4), slot_writes=(0, 4), allow_new_accounts=False, allow_self_destruct=False)
    want = oracle.block_decode(blk.flat)
    assert ctx.block_decode(blk.flat) == want
    st = ctx.stats()
    assert st["txn_loops_on_gpu"] == 1 and st["marks_on_gpu"] > 12 * 20
    for seed in (1, 2, 3):  # config-1 shaped blocks with new accounts, self-destructs, withdrawals
        c1 = synth.gen_block(seed, n_accounts=1000, n_txns=10, n_withdrawals=seed % 3)
        assert ctx.block_decode(c1.flat) == oracle.block_decode(c1.flat)
        assert ctx.stats()["marks_on_gpu"] > 0
    # a new account in a state with hashed-out siblings: its key runs into a hash node
    bad = synth.gen_block(78, n_accounts=300, n_txns=4, virtual_depth=3, virtual_accounts_log16=5, accounts_per_txn=(5, 10),
                          allow_new_accounts=True, allow_self_destruct=False)
    try:
        want_bad = oracle.block_decode(bad.flat)
    except OracleError as e:
        with pytest.raises(Exception) as ei:
            ctx.block_decode(bad.flat)
        assert getattr(ei.value, "code", None) == e.code
        assert ctx.stats()["txn_loops_on_gpu"] == 0  # the host path reported it
    else:
        assert ctx.block_decode(bad.flat) == want_bad
