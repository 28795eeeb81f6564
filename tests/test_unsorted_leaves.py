"""ppd_trie_root_leaves[_dev]: trie roots from leaves in any order, with repeated keys (the last value wins) and keys
that are hashed first (PPD_LEAVES_HASH_KEYS).

Where it matters a root is checked three ways: the new entry, the oracle inserting the leaves in input order
(oracle_trie_root_from_leaves), and the sorted entry on a numpy sort-and-dedupe of the leaves.
"""
import numpy as np
import pytest

from test_node_encoding_edges import _arrays, _model_root, gadgets, union

BAD_ARGUMENT = 62


@pytest.fixture(scope="module")
def ctx():
    from proof_protocol_decoder_b200.lib import Context

    c = Context(0)
    yield c
    c.close()


# ---------------------------------------------------------------- helpers -------------------------------------------
def pack(values):
    """[bytes] -> (val_off uint64 [n+1], vals uint8)"""
    off = np.zeros(len(values) + 1, dtype=np.uint64)
    np.cumsum([len(v) for v in values], out=off[1:])
    vals = np.frombuffer(b"".join(values) or b"\0", dtype=np.uint8)[: int(off[-1])].copy()
    return off, vals


def values_of(off, vals):
    return [bytes(vals[int(off[i]) : int(off[i + 1])]) for i in range(len(off) - 1)]


def permute(keys, off, vals, perm):
    v = values_of(off, vals)
    o, pool = pack([v[i] for i in perm])
    return np.ascontiguousarray(keys[perm]), o, pool


def sort_dedupe(keys, off, vals):
    """numpy reference of the contract: sort by key, keep the last occurrence of each key"""
    n = len(keys)
    if n == 0:
        return keys.reshape(0, 32), np.zeros(1, np.uint64), np.zeros(0, np.uint8)
    be = np.ascontiguousarray(keys).view(">u8")
    order = np.lexsort((np.arange(n), be[:, 3], be[:, 2], be[:, 1], be[:, 0]))
    k = keys[order]
    last = np.ones(n, dtype=bool)
    last[:-1] = (k[1:] != k[:-1]).any(axis=1)
    keep = order[last]
    v = values_of(off, vals)
    o, pool = pack([v[i] for i in keep])
    return np.ascontiguousarray(keys[keep]), o, pool


def three_way(ctx, oracle, keys, off, vals):
    got = ctx.trie_root_leaves(keys, off, vals)
    assert got == oracle.trie_root_from_leaves(keys, off, vals), "new entry vs the oracle inserting in input order"
    assert got == ctx.trie_root_sorted_leaves(*sort_dedupe(keys, off, vals)), "new entry vs the sorted entry on the deduplicated set"
    return got


def rand_values(rng, n, lo=1, hi=40):
    return [rng.bytes(int(x)) for x in rng.integers(lo, hi + 1, size=n)]


def shuffled_sorted_leaves(n, seed):
    from proof_protocol_decoder_b200 import synth

    keys, off, vals = synth.gen_sorted_leaves(n, seed=seed)
    perm = np.random.default_rng(seed).permutation(n)
    return permute(keys, off, vals, perm)


def gadget_arrays(items, seed):
    keys, off, vals = _arrays(items)
    return permute(keys, off, vals, np.random.default_rng(seed).permutation(len(items)))


def hashed(oracle, keys):
    n, kl = keys.shape
    return oracle.keccak256_batch(keys.reshape(-1), np.arange(n + 1, dtype=np.uint64) * kl)


# ---------------------------------------------------------------- CPU -----------------------------------------------
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_sort_dedupe_helper_matches_insertion_order(oracle, seed):
    rng = np.random.default_rng(seed)
    pool = np.frombuffer(rng.bytes(32 * 300), dtype=np.uint8).reshape(300, 32)
    keys = np.ascontiguousarray(pool[rng.integers(0, 300, size=1000)])
    off, vals = pack(rand_values(rng, 1000))
    assert len(np.unique(keys, axis=0)) < 1000
    assert oracle.trie_root_from_leaves(keys, off, vals) == oracle.trie_root_from_leaves(*sort_dedupe(keys, off, vals))


# ---------------------------------------------------------------- order and size ------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 2, 3, 17, 1000, 50_000, 1_000_000])
def test_shuffled_distinct_keys(ctx, oracle, n):
    keys, off, vals = shuffled_sorted_leaves(n, seed=n + 7)
    three_way(ctx, oracle, keys, off, vals)


# ---------------------------------------------------------------- duplicates ----------------------------------------
@pytest.mark.gpu
def test_adjacent_and_distant_repeats_keep_the_last_value(ctx, oracle):
    rng = np.random.default_rng(11)
    base = np.frombuffer(rng.bytes(32 * 500), dtype=np.uint8).reshape(500, 32)
    rows = list(range(500))
    rows[10:10] = [10, 10]  # adjacent repeats
    rows += [3, 250, 499, 0]  # distant repeats
    keys = np.ascontiguousarray(base[rows])
    off, vals = pack(rand_values(rng, len(rows)))
    root = three_way(ctx, oracle, keys, off, vals)
    first_wins = sort_dedupe(keys[::-1].copy(), *pack(values_of(off, vals)[::-1]))
    assert root != ctx.trie_root_sorted_leaves(*first_wins)


@pytest.mark.gpu
def test_every_key_repeated(ctx, oracle):
    rng = np.random.default_rng(12)
    base = np.frombuffer(rng.bytes(32 * 2000), dtype=np.uint8).reshape(2000, 32)
    rows = rng.permutation(np.concatenate([np.arange(2000)] * 3))
    keys = np.ascontiguousarray(base[rows])
    off, vals = pack(rand_values(rng, len(rows)))
    three_way(ctx, oracle, keys, off, vals)


@pytest.mark.gpu
def test_ten_thousand_copies_of_one_key_are_one_leaf(ctx, oracle):
    rng = np.random.default_rng(13)
    key = np.frombuffer(rng.bytes(32), dtype=np.uint8)
    keys = np.ascontiguousarray(np.tile(key, (10_000, 1)))
    values = rand_values(rng, 10_000)
    off, vals = pack(values)
    root = three_way(ctx, oracle, keys, off, vals)
    assert root == ctx.trie_root_sorted_leaves(key.reshape(1, 32).copy(), *pack([values[-1]]))


@pytest.mark.gpu
def test_final_value_equal_to_an_earlier_one(ctx, oracle):
    rng = np.random.default_rng(14)
    base = np.frombuffer(rng.bytes(32 * 50), dtype=np.uint8).reshape(50, 32)
    values = rand_values(rng, 50)
    keys = np.ascontiguousarray(np.concatenate([base, base[7:8], base[7:8]]))
    off, vals = pack(values + [b"\x01\x02\x03", values[7]])
    root = three_way(ctx, oracle, keys, off, vals)
    assert root == ctx.trie_root_sorted_leaves(*sort_dedupe(base.copy(), *pack(values)))


# ---------------------------------------------------------------- tie refinement at every word boundary -------------
def _boundary_keys(rng):
    base = np.frombuffer(rng.bytes(32), dtype=np.uint8)
    rows = []
    for b in (8, 16, 24):  # equal in the first b bytes, different in byte b
        for v in range(0, 256, 37):
            k = np.frombuffer(rng.bytes(32), dtype=np.uint8).copy()
            k[:b] = base[:b]
            k[b] = v
            rows.append(k)
    for nib in range(16):  # equal but for the last nibble
        k = base.copy()
        k[31] = (k[31] & 0xF0) | nib
        rows.append(k)
    return np.array(rows, dtype=np.uint8)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [21, 22])
def test_keys_tied_up_to_each_word_boundary(ctx, oracle, seed):
    rng = np.random.default_rng(seed)
    distinct = _boundary_keys(rng)
    rows = rng.permutation(np.concatenate([np.arange(len(distinct)), rng.integers(0, len(distinct), size=40)]))
    keys = np.ascontiguousarray(distinct[rows])
    off, vals = pack(rand_values(rng, len(rows)))
    three_way(ctx, oracle, keys, off, vals)


@pytest.mark.gpu
def test_shared_prefix_set_shuffled(ctx, oracle):
    # the key set of test_gpu_parity.py::test_sorted_leaves_shared_prefixes_and_small_values, in a random order
    rng = np.random.default_rng(3)
    n = 4000
    keys = np.zeros((n, 32), dtype=np.uint8)
    keys[:, :28] = np.frombuffer(rng.bytes(28), dtype=np.uint8)
    keys[:, 28:] = np.frombuffer(rng.bytes(4 * n), dtype=np.uint8).reshape(n, 4)
    keys[: n // 2, 5] ^= 0x10
    keys = np.unique(keys, axis=0)
    n = len(keys)
    off, vals = pack(rand_values(rng, n, 1, 3))
    keys, off, vals = permute(keys, off, vals, rng.permutation(n))
    three_way(ctx, oracle, keys, off, vals)


# ---------------------------------------------------------------- node-encoding gadgets -----------------------------
@pytest.mark.gpu
def test_every_gadget_shuffled(ctx, oracle):
    for g, (name, items) in enumerate(gadgets("raw")):
        arrays = gadget_arrays(items, g)
        want = _model_root(items)
        assert ctx.trie_root_leaves(*arrays) == want, name
        assert oracle.trie_root_from_leaves(*arrays) == want, name


@pytest.mark.gpu
def test_all_gadgets_at_once_shuffled(ctx, oracle):
    items = union("raw")
    arrays = gadget_arrays(items, 99)
    assert three_way(ctx, oracle, *arrays) == _model_root(items)


# ---------------------------------------------------------------- hashed keys ---------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("key_len", [20, 32])
def test_hashed_addresses_and_slots_with_repeats(ctx, oracle, key_len):
    rng = np.random.default_rng(key_len)
    pool = np.frombuffer(rng.bytes(key_len * 3000), dtype=np.uint8).reshape(3000, key_len)
    raw = np.ascontiguousarray(pool[rng.integers(0, 3000, size=5000)])
    off, vals = pack(rand_values(rng, 5000, 2, 90))
    root = ctx.trie_root_leaves(raw, off, vals, hash_keys=True)
    st = ctx.stats()
    assert st["key_hashes"] == 5000 and st["key_permutations"] == 5000
    h = hashed(oracle, raw)
    assert root == oracle.trie_root_from_leaves(h, off, vals)
    assert root == ctx.trie_root_leaves(h, off, vals)


@pytest.mark.gpu
@pytest.mark.parametrize("key_len", [1, 135])
def test_hashed_key_length_limits(ctx, oracle, key_len):
    rng = np.random.default_rng(key_len + 1000)
    n = 300 if key_len == 1 else 2000
    raw = np.frombuffer(rng.bytes(key_len * n), dtype=np.uint8).reshape(n, key_len).copy()
    off, vals = pack(rand_values(rng, n))
    root = ctx.trie_root_leaves(raw, off, vals, hash_keys=True)
    assert root == oracle.trie_root_from_leaves(hashed(oracle, raw), off, vals)


@pytest.mark.gpu
def test_bad_key_lengths_and_flags_are_rejected(ctx):
    import torch

    from proof_protocol_decoder_b200 import PpdError

    rng = np.random.default_rng(5)
    off, vals = pack(rand_values(rng, 4))
    for key_len, hash_keys in ((0, True), (136, True), (20, False), (33, False)):
        keys = np.frombuffer(rng.bytes(4 * key_len), dtype=np.uint8).reshape(4, key_len).copy()
        with pytest.raises(PpdError) as e:
            ctx.trie_root_leaves(keys, off, vals, hash_keys=hash_keys)
        assert e.value.code == BAD_ARGUMENT, (key_len, hash_keys)
    keys = torch.zeros((4, 32), dtype=torch.uint8, device="cuda")
    d_off = torch.from_numpy(off.astype(np.int64)).cuda()
    d_vals = torch.from_numpy(vals).cuda()
    torch.cuda.synchronize()
    for flags in (2, 0x80000000, 3):
        with pytest.raises(PpdError) as e:
            ctx.trie_root_leaves_dev(keys.data_ptr(), 32, d_off.data_ptr(), d_vals.data_ptr(), 4, d_vals.numel(), flags=flags)
        assert e.value.code == BAD_ARGUMENT, flags


# ---------------------------------------------------------------- bad offsets, inputs untouched, alignment ----------
def _dev(keys, off, vals, pad=0):
    import torch

    return (torch.from_numpy(np.ascontiguousarray(keys)).cuda(), torch.from_numpy(off.astype(np.int64)).cuda(),
            torch.from_numpy(np.concatenate([vals, np.zeros(pad, np.uint8)])).cuda())


def _root_dev(ctx, k, o, v, n=None, vals_bytes=None, hash_keys=False):
    import torch

    torch.cuda.synchronize()  # the library reads the buffers on a stream of its own
    n = o.numel() - 1 if n is None else n
    return ctx.trie_root_leaves_dev(k.data_ptr(), k.shape[1], o.data_ptr(), v.data_ptr(), n, v.numel() if vals_bytes is None else vals_bytes,
                                    hash_keys=hash_keys)


@pytest.mark.gpu
def test_bad_offsets_are_rejected(ctx):
    from proof_protocol_decoder_b200 import PpdError

    keys, off, vals = shuffled_sorted_leaves(1000, seed=31)
    k, o, v = _dev(keys, off, vals)
    good = _root_dev(ctx, k, o, v)
    dec = o.clone()
    dec[500] = dec[499] - 1  # decreasing once
    big = o.clone()
    big[-1] = v.numel() + 1  # past the readable bytes
    for bad in (dec, big):
        with pytest.raises(PpdError) as e:
            _root_dev(ctx, k, bad, v)
        assert e.value.code == BAD_ARGUMENT
    with pytest.raises(PpdError) as e:
        _root_dev(ctx, k, o, v, vals_bytes=v.numel() - 1)
    assert e.value.code == BAD_ARGUMENT
    dec_host = off.copy()
    dec_host[10] = dec_host[9] - np.uint64(1)
    with pytest.raises(PpdError) as e:
        ctx.trie_root_leaves(keys, dec_host, vals)
    assert e.value.code == BAD_ARGUMENT
    assert _root_dev(ctx, k, o, v) == good  # the context still works


@pytest.mark.gpu
@pytest.mark.parametrize("hash_keys", [False, True])
def test_inputs_are_untouched(ctx, hash_keys):
    keys, off, vals = shuffled_sorted_leaves(20_000, seed=41)
    keys[100:200] = keys[0]  # repeats: every stage runs
    if hash_keys:
        keys = np.ascontiguousarray(keys[:, :20])
    k, o, v = _dev(keys, off, vals)
    before = [t.clone() for t in (k, o, v)]
    _root_dev(ctx, k, o, v, hash_keys=hash_keys)
    for a, b in zip(before, (k, o, v)):
        assert bool((a == b).all())


@pytest.mark.gpu
def test_value_alignment(ctx, oracle):
    import torch

    keys, off, vals = shuffled_sorted_leaves(30_000, seed=51)
    want = three_way(ctx, oracle, keys[:3000].copy(), off[:3001].copy(), vals[: int(off[3000])].copy())
    k, o, v = _dev(keys[:3000], off[:3001], vals[: int(off[3000])])
    for shift in (1, 2, 3):
        shifted = torch.cat([torch.full((shift,), 0xEE, dtype=torch.uint8, device="cuda"), v])
        assert _root_dev(ctx, k, o + shift, shifted) == want, shift
    flipped = v.clone()
    flipped[int(off[1234]) + 5] ^= 0x04
    assert _root_dev(ctx, k, o, flipped) != want


# ---------------------------------------------------------------- buffer reuse, host vs device, stats ---------------
@pytest.mark.gpu
def test_buffer_reuse_and_host_device_agree(ctx):
    big = shuffled_sorted_leaves(1_000_000, seed=61)
    small = shuffled_sorted_leaves(3, seed=62)
    want_big = ctx.trie_root_sorted_leaves(*sort_dedupe(*big))
    want_small = ctx.trie_root_sorted_leaves(*sort_dedupe(*small))
    for arrays, want in ((big, want_big), (small, want_small), (big, want_big)):
        assert ctx.trie_root_leaves(*arrays) == want
        assert _root_dev(ctx, *_dev(*arrays)) == want


@pytest.mark.gpu
def test_stats_match_the_sorted_entry(ctx):
    rng = np.random.default_rng(71)
    keys, off, vals = shuffled_sorted_leaves(50_000, seed=71)
    rows = rng.integers(0, 50_000, size=60_000)
    keys, off, vals = permute(keys, off, vals, rows)
    ctx.trie_root_sorted_leaves(*sort_dedupe(keys, off, vals))
    want = ctx.stats()
    ctx.trie_root_leaves(keys, off, vals)
    got = ctx.stats()
    for f in ("nodes_hashed", "node_permutations", "node_bytes", "arena_nodes", "levels"):
        assert got[f] == want[f], f
    assert got["key_hashes"] == 0
    assert got["gpu_ms"] > 0 and got["kernel_launches"] > want["kernel_launches"]


# ---------------------------------------------------------------- scale ---------------------------------------------
@pytest.mark.gpu
def test_ten_million_device_leaves_permuted(ctx):
    import torch

    from proof_protocol_decoder_b200 import synth

    n = 10_000_000
    keys, off, vals = synth.gen_sorted_leaves_dev(n, seed=81)
    torch.cuda.synchronize()  # the library reads the buffers on a stream of its own
    want = ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel())
    assert ctx.trie_root_leaves_dev(keys.data_ptr(), 32, off.data_ptr(), vals.data_ptr(), n, vals.numel()) == want
    g = torch.Generator(device="cuda")
    g.manual_seed(82)
    pk, po, pv = synth.permute_leaves_dev(keys, off, vals, torch.randperm(n, generator=g, device="cuda"))
    del keys, off, vals
    torch.cuda.synchronize()
    assert ctx.trie_root_leaves_dev(pk.data_ptr(), 32, po.data_ptr(), pv.data_ptr(), n, pv.numel()) == want
