"""ppd_trie_subset_[sorted_]leaves[_dev]: create_trie_subset of the trie over leaves, cut on the GPU.

Three references: a pure-Python subset over trie_model (here), the CPU oracle's create_trie_subset (exported for these
tests by tests/cpp/trie_subset_oracle.cpp, which includes oracle/ppd_oracle.cpp) and, for whole pre-images, the GPU witness parser and level hasher, which share no code
with the builder: a subset wrapped as a DirectPreImage must hash to the trie's root.
"""
import collections

import numpy as np
import pytest

import trie_model as tm
from test_node_encoding_edges import _arrays, _bytes_key, gadgets, union
from test_unsorted_leaves import _dev, pack, permute, rand_values, shuffled_sorted_leaves, sort_dedupe

BAD_ARGUMENT, UNSORTED_KEYS = 62, 63


@pytest.fixture(scope="module")
def ctx():
    from proof_protocol_decoder_b200.lib import Context

    c = Context(0)
    yield c
    c.close()


class SubsetOracle:
    """The session oracle plus trie_subset_from_leaves, from tests/cpp/trie_subset_oracle.cpp"""

    def __init__(self, base, so_path):
        import ctypes

        self.base = base
        self.L = ctypes.CDLL(str(so_path))
        u8p = ctypes.POINTER(ctypes.c_uint8)
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        self.L.oracle_trie_subset_from_leaves.argtypes = [vp, vp, vp, sz, vp, sz, ctypes.POINTER(u8p), ctypes.POINTER(sz), ctypes.c_char_p, sz]
        self.L.oracle_free.argtypes = [vp]

    def __getattr__(self, name):
        return getattr(self.base, name)

    def trie_subset_from_leaves(self, keys, val_off, vals, queries) -> bytes:
        """create_trie_subset of the trie over the leaves (inserted in input order) for 32-byte queries: one Trie in the
        pre-order Node form of include/ppd_flat.h"""
        import ctypes

        from ppd_oracle_lib import OracleError

        keys = np.ascontiguousarray(keys, dtype=np.uint8)
        val_off = np.ascontiguousarray(val_off, dtype=np.uint64)
        vals = np.ascontiguousarray(vals, dtype=np.uint8)
        queries = np.ascontiguousarray(queries, dtype=np.uint8).reshape(-1, 32)
        out, n = ctypes.POINTER(ctypes.c_uint8)(), ctypes.c_size_t()
        err = ctypes.create_string_buffer(512)
        rc = self.L.oracle_trie_subset_from_leaves(keys.ctypes.data, val_off.ctypes.data, vals.ctypes.data, len(val_off) - 1, queries.ctypes.data,
                                                   len(queries), ctypes.byref(out), ctypes.byref(n), err, 512)
        if rc:
            raise OracleError(rc, err.value.decode(errors="replace"))
        res = ctypes.string_at(out, n.value)
        self.L.oracle_free(out)
        return res


@pytest.fixture(scope="module")
def subset_oracle(oracle, tmp_path_factory):
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = tmp_path_factory.mktemp("subset_oracle") / "libtrie_subset_oracle.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), os.path.join(root, "tests", "cpp", "trie_subset_oracle.cpp")])
    return SubsetOracle(oracle, so)


# ---------------------------------------------------------------- the model -----------------------------------------
def model_subset(items, queries, stops=None):
    """create_trie_subset over sorted model items [(64 nibbles, value)] for query nibble lists -> node tuple (flat.encode_node).
    A node no query reaches is ("hash", keccak(rlp)) when its RLP has 32 bytes or more, else written whole.  `stops`
    (a Counter) counts where absent queries leave the trie: "leaf", "empty", ("ext", parity of the nibble that differs)."""
    stops = collections.Counter() if stops is None else stops

    def node(its, depth, qs):
        if not qs:
            raw = tm.node_rlp(its, depth)
            if len(raw) >= 32:
                return ("hash", tm.keccak(raw))
        if len(its) == 1:
            nib, val = its[0]
            stops["leaf"] += sum(q != nib for q in qs)
            return ("leaf", nib[depth:], val)
        cp = tm.common_depth(its, depth)
        if cp > depth:
            ext = its[0][0][depth:cp]
            on = []
            for q in qs:
                if q[depth:cp] == ext:
                    on.append(q)
                else:
                    p = next(i for i in range(depth, cp) if q[i] != ext[i - depth])
                    stops[("ext", p & 1)] += 1
            return ("extension", ext, node(its, cp, on))
        kids = tm.split_children(its, depth)
        ch = []
        for s in range(16):
            on = [q for q in qs if q[depth] == s]
            if kids[s]:
                ch.append(node(kids[s], depth + 1, on))
            else:
                stops["empty"] += len(on)
                ch.append(("empty",))
        return ("branch", ch, b"")

    if not items:
        return ("empty",)
    return node(items, 0, [list(q) for q in queries])


def items_of_arrays(keys, off, vals):
    """the model items of the trie the leaves give (sorted, the last value of a repeated key)"""
    k, o, v = sort_dedupe(np.ascontiguousarray(keys), off, vals)
    return [(tm.nibbles(bytes(k[i])), bytes(v[int(o[i]) : int(o[i + 1])])) for i in range(len(k))]


def nibbles_of(q):
    return [tm.nibbles(bytes(r)) for r in np.asarray(q, dtype=np.uint8).reshape(-1, 32)]


def probes(keys, rng, n_keys=4):
    """keys one nibble away from present keys, at every position 0..63: they leave the trie at an empty slot, inside an
    extension, at a leaf with another suffix, or (when the changed key exists) are present"""
    out = []
    for r in rng.choice(len(keys), size=min(n_keys, len(keys)), replace=False):
        nib = tm.nibbles(bytes(keys[r]))
        for p in range(64):
            q = list(nib)
            q[p] = (q[p] + 1 + int(rng.integers(0, 15))) % 16
            out.append(list(_bytes_key(q)))
    return np.array(out, dtype=np.uint8).reshape(-1, 32)


def mixed_queries(keys, m, rng):
    """m queries: half present keys, half random (absent) keys, a few repeated"""
    present = keys[rng.integers(0, len(keys), size=m - m // 2)] if len(keys) else np.zeros((0, 32), np.uint8)
    absent = np.frombuffer(rng.bytes(32 * (m // 2)), dtype=np.uint8).reshape(-1, 32)
    q = np.concatenate([present.reshape(-1, 32), absent])
    return np.ascontiguousarray(q[rng.permutation(len(q))])


def structured_set(rng, n=600):
    """random keys plus clusters sharing prefixes of every length: extensions of both parities everywhere"""
    keys = [rng.bytes(32) for _ in range(n)]
    for L in range(1, 63, 3):
        base = tm.nibbles(rng.bytes(32))
        for _ in range(3):
            tail = tm.nibbles(rng.bytes(32))
            keys.append(_bytes_key(base[:L] + tail[L:]))
    keys = np.unique(np.frombuffer(b"".join(keys), dtype=np.uint8).reshape(-1, 32), axis=0)
    off, vals = pack(rand_values(rng, len(keys), 1, 40))
    return keys, off, vals


# ---------------------------------------------------------------- CPU: the model against the oracle -----------------
def _model_vs_oracle(subset_oracle, keys, off, vals, queries, stops=None):
    from proof_protocol_decoder_b200 import flat

    want = subset_oracle.trie_subset_from_leaves(keys, off, vals, queries)
    got = model_subset(items_of_arrays(keys, off, vals), nibbles_of(queries), stops)
    assert flat.parse_trie(want) == got
    assert flat.encode_node(got) == want
    return want


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_model_equals_oracle_on_random_sets(subset_oracle, seed):
    rng = np.random.default_rng(seed)
    keys, off, vals = structured_set(rng)
    stops = collections.Counter()
    q = np.concatenate([probes(keys, rng, 40), mixed_queries(keys, 200, rng), keys[:5], keys[:5]])
    _model_vs_oracle(subset_oracle, keys, off, vals, q, stops)
    assert stops["leaf"] and stops["empty"] and stops[("ext", 0)] and stops[("ext", 1)], stops
    _model_vs_oracle(subset_oracle, keys, off, vals, np.zeros((0, 32), np.uint8))
    _model_vs_oracle(subset_oracle, keys, off, vals, keys)


def test_model_equals_oracle_on_every_gadget(subset_oracle):
    items = union("raw")
    keys, off, vals = _arrays(items)
    for name, its in gadgets("raw"):
        mine = {tuple(k) for k, _ in its}
        own = np.array([list(_bytes_key(k)) for k, _ in its], dtype=np.uint8)
        others = np.array([list(_bytes_key(k)) for k, _ in items if tuple(k) not in mine], dtype=np.uint8)
        gk, go, gv = _arrays(its)
        _model_vs_oracle(subset_oracle, gk, go, gv, own)
        _model_vs_oracle(subset_oracle, gk, go, gv, probes(own, np.random.default_rng(len(name)), 2))
        _model_vs_oracle(subset_oracle, keys, off, vals, others)


def test_model_equals_oracle_small_and_empty(subset_oracle):
    rng = np.random.default_rng(9)
    none = np.zeros((0, 32), np.uint8)
    e_keys, e_off, e_vals = np.zeros((0, 32), np.uint8), np.zeros(1, np.uint64), np.zeros(0, np.uint8)
    assert _model_vs_oracle(subset_oracle, e_keys, e_off, e_vals, none) == bytes([0])
    assert _model_vs_oracle(subset_oracle, e_keys, e_off, e_vals, mixed_queries(e_keys, 4, rng)) == bytes([0])
    one = np.frombuffer(rng.bytes(32), dtype=np.uint8).reshape(1, 32).copy()
    o1, v1 = pack([b"\x01\x02\x03"])
    for q in (none, one, probes(one, rng, 1), mixed_queries(one, 6, rng)):
        _model_vs_oracle(subset_oracle, one, o1, v1, q)
    assert _model_vs_oracle(subset_oracle, one, o1, v1, none)[0] == 1  # the untouched root is HASH(root)


# ---------------------------------------------------------------- GPU ----------------------------------------------
def _check(ctx, subset_oracle, keys, off, vals, queries, model=True, sorted_entry=True):
    """the any-order entry against the oracle (and the model up to 10 k leaves), the sorted entry on the numpy
    sort-and-dedupe, and the roots of the root entries"""
    root, got = ctx.trie_subset_leaves(keys, off, vals, queries)
    assert root == ctx.trie_root_leaves(keys, off, vals)
    assert got == subset_oracle.trie_subset_from_leaves(keys, off, vals, queries), "GPU subset vs the oracle"
    if model and len(keys) <= 10_000:
        from proof_protocol_decoder_b200 import flat

        assert flat.parse_trie(got) == model_subset(items_of_arrays(keys, off, vals), nibbles_of(queries))
    if sorted_entry:
        sk, so, sv = sort_dedupe(keys, off, vals)
        assert _sorted_dev(ctx, sk, so, sv, queries) == (root, got)
    return root, got


def _sorted_dev(ctx, keys, off, vals, queries):
    import torch

    k, o, v = _dev(keys, off, vals)
    q = torch.from_numpy(np.ascontiguousarray(queries, dtype=np.uint8).reshape(-1, 32)).cuda()
    torch.cuda.synchronize()
    return ctx.trie_subset_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), len(keys), v.numel(), q.data_ptr(), q.shape[0])


@pytest.mark.gpu
@pytest.mark.parametrize("n,m", [(1000, 1), (1000, 1000), (1000, 100_000), (100_000, 1), (100_000, 1000), (100_000, 100_000),
                                 (1_000_000, 1), (1_000_000, 1000), (1_000_000, 100_000)])
def test_random_sets(ctx, subset_oracle, n, m):
    rng = np.random.default_rng(n + m)
    keys, off, vals = shuffled_sorted_leaves(n, seed=n + 3)
    _check(ctx, subset_oracle, keys, off, vals, mixed_queries(keys, m, rng))


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [4, 5])
def test_every_divergence_and_repeat(ctx, subset_oracle, seed):
    rng = np.random.default_rng(seed)
    keys, off, vals = structured_set(rng, 3000)
    keys, off, vals = permute(keys, off, vals, rng.permutation(len(keys)))
    q = np.concatenate([probes(keys, rng, 16), mixed_queries(keys, 500, rng)])
    q = np.concatenate([q, q[::7]])
    _check(ctx, subset_oracle, keys, off, vals, q)
    _check(ctx, subset_oracle, keys, off, vals, np.zeros((0, 32), np.uint8))


@pytest.mark.gpu
def test_all_keys_queried_is_the_whole_trie(ctx, subset_oracle):
    from proof_protocol_decoder_b200 import flat

    keys, off, vals = shuffled_sorted_leaves(5000, seed=17)
    _, got = _check(ctx, subset_oracle, keys, off, vals, keys)

    def kinds(t):
        yield t[0]
        if t[0] == "branch":
            for c in t[1]:
                yield from kinds(c)
        elif t[0] == "extension":
            yield from kinds(t[2])

    k = collections.Counter(kinds(flat.parse_trie(got)))
    assert k["hash"] == 0 and k["leaf"] == 5000, k


@pytest.mark.gpu
def test_no_queries_and_tiny_tries(ctx, subset_oracle):
    rng = np.random.default_rng(23)
    none = np.zeros((0, 32), np.uint8)
    keys, off, vals = shuffled_sorted_leaves(3000, seed=23)
    root, got = _check(ctx, subset_oracle, keys, off, vals, none)
    assert got == bytes([1]) + root
    e = (np.zeros((0, 32), np.uint8), np.zeros(1, np.uint64), np.zeros(0, np.uint8))
    assert ctx.trie_subset_leaves(*e, mixed_queries(e[0], 3, rng)) == (tm.EMPTY_TRIE_HASH, bytes([0]))
    assert ctx.trie_subset_leaves(*e, none) == (tm.EMPTY_TRIE_HASH, bytes([0]))
    for n in (1, 2, 3):
        k, o, v = shuffled_sorted_leaves(n, seed=n)
        for q in (none, k, probes(k, rng, 1), mixed_queries(k, 5, rng)):
            _check(ctx, subset_oracle, k, o, v, q)


@pytest.mark.gpu
def test_every_gadget_own_keys_and_neighbours(ctx, subset_oracle):
    items = union("raw")
    keys, off, vals = _arrays(items)
    for g, (name, its) in enumerate(gadgets("raw")):
        mine = {tuple(k) for k, _ in its}
        own = np.array([list(_bytes_key(k)) for k, _ in its], dtype=np.uint8)
        others = np.array([list(_bytes_key(k)) for k, _ in items if tuple(k) not in mine], dtype=np.uint8)
        gk, go, gv = _arrays(its)
        gk, go, gv = permute(gk, go, gv, np.random.default_rng(g).permutation(len(gk)))
        _check(ctx, subset_oracle, gk, go, gv, own)
        _check(ctx, subset_oracle, gk, go, gv, probes(own, np.random.default_rng(g), 2))
        _check(ctx, subset_oracle, keys, off, vals, others)


@pytest.mark.gpu
def test_repeated_leaves_equal_the_sorted_entry(ctx, subset_oracle):
    rng = np.random.default_rng(29)
    base = np.frombuffer(rng.bytes(32 * 3000), dtype=np.uint8).reshape(3000, 32)
    keys = np.ascontiguousarray(base[rng.integers(0, 3000, size=8000)])
    off, vals = pack(rand_values(rng, 8000))
    _check(ctx, subset_oracle, keys, off, vals, np.concatenate([mixed_queries(keys, 2000, rng), probes(keys, rng, 4)]))


@pytest.mark.gpu
@pytest.mark.parametrize("key_len", [20, 32])
def test_hashed_keys_and_queries(ctx, subset_oracle, key_len):
    from test_unsorted_leaves import hashed

    rng = np.random.default_rng(key_len + 1)
    pool = np.frombuffer(rng.bytes(key_len * 4000), dtype=np.uint8).reshape(4000, key_len)
    raw = np.ascontiguousarray(pool[rng.integers(0, 4000, size=5000)])
    off, vals = pack(rand_values(rng, 5000, 2, 90))
    rq = np.ascontiguousarray(np.concatenate([raw[:300], np.frombuffer(rng.bytes(key_len * 300), dtype=np.uint8).reshape(300, key_len)]))
    root, got = ctx.trie_subset_leaves(raw, off, vals, rq, hash_keys=True)
    st = ctx.stats()
    assert st["key_hashes"] == 5000 + 600
    hk, hq = hashed(subset_oracle, raw), hashed(subset_oracle, rq)
    assert (root, got) == ctx.trie_subset_leaves(hk, off, vals, hq)
    assert got == subset_oracle.trie_subset_from_leaves(hk, off, vals, hq)
    import torch

    k, o, v = _dev(raw, off, vals)
    q = torch.from_numpy(rq).cuda()
    torch.cuda.synchronize()
    assert ctx.trie_subset_leaves_dev(k.data_ptr(), key_len, o.data_ptr(), v.data_ptr(), 5000, v.numel(), q.data_ptr(), 600, hash_keys=True) == (root, got)


@pytest.mark.gpu
def test_argument_checks(ctx):
    import torch

    from proof_protocol_decoder_b200 import PpdError

    rng = np.random.default_rng(31)
    keys, off, vals = shuffled_sorted_leaves(100, seed=31)
    q = keys[:3].copy()
    for key_len, hash_keys in ((0, True), (136, True), (20, False)):
        kk = np.frombuffer(rng.bytes(100 * key_len), dtype=np.uint8).reshape(100, key_len).copy()
        with pytest.raises(PpdError) as e:
            ctx.trie_subset_leaves(kk, off, vals, kk[:2], hash_keys=hash_keys)
        assert e.value.code == BAD_ARGUMENT
    k, o, v = _dev(keys, off, vals)
    dq = torch.from_numpy(q).cuda()
    torch.cuda.synchronize()
    for flags in (2, 3):
        with pytest.raises(PpdError) as e:
            ctx.trie_subset_leaves_dev(k.data_ptr(), 32, o.data_ptr(), v.data_ptr(), 100, v.numel(), dq.data_ptr(), 3, flags=flags)
        assert e.value.code == BAD_ARGUMENT
    bad = o.clone()
    bad[50] = bad[49] - 1
    with pytest.raises(PpdError) as e:
        ctx.trie_subset_leaves_dev(k.data_ptr(), 32, bad.data_ptr(), v.data_ptr(), 100, v.numel(), dq.data_ptr(), 3)
    assert e.value.code == BAD_ARGUMENT
    for m in (0x7FFFFFFE, 1 << 40):
        with pytest.raises(PpdError) as e:
            ctx.trie_subset_leaves_dev(k.data_ptr(), 32, o.data_ptr(), v.data_ptr(), 100, v.numel(), dq.data_ptr(), m)
        assert e.value.code == BAD_ARGUMENT
        with pytest.raises(PpdError) as e:
            ctx.trie_subset_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), 100, v.numel(), dq.data_ptr(), m)
        assert e.value.code == BAD_ARGUMENT
    with pytest.raises(PpdError) as e:
        ctx.trie_subset_leaves_dev(k.data_ptr(), 32, o.data_ptr(), v.data_ptr(), 0x7FFFFFFF, v.numel(), dq.data_ptr(), 3)
    assert e.value.code == BAD_ARGUMENT
    with pytest.raises(PpdError) as e:  # any order given to the sorted entry
        ctx.trie_subset_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), 100, v.numel(), dq.data_ptr(), 3)
    assert e.value.code == UNSORTED_KEYS
    want = ctx.trie_subset_leaves(keys, off, vals, q)
    assert ctx.trie_subset_leaves_dev(k.data_ptr(), 32, o.data_ptr(), v.data_ptr(), 100, v.numel(), dq.data_ptr(), 3) == want  # still works


@pytest.mark.gpu
def test_inputs_untouched_buffer_reuse_host_and_device_agree(ctx):
    import torch

    rng = np.random.default_rng(37)
    big = shuffled_sorted_leaves(1_000_000, seed=37)
    small = shuffled_sorted_leaves(50, seed=38)
    runs = []
    for keys, off, vals in (big, small, big):
        q = mixed_queries(keys, 20_000 if len(keys) > 50 else 30, rng)
        want = ctx.trie_subset_leaves(keys, off, vals, q)
        k, o, v = _dev(keys, off, vals)
        dq = torch.from_numpy(q).cuda()
        before = [t.clone() for t in (k, o, v, dq)]
        torch.cuda.synchronize()
        got = ctx.trie_subset_leaves_dev(k.data_ptr(), 32, o.data_ptr(), v.data_ptr(), len(keys), v.numel(), dq.data_ptr(), len(q))
        assert got == want
        for a, b in zip(before, (k, o, v, dq)):
            assert bool((a == b).all())
        runs.append(want)
    st = ctx.stats()
    assert st["gpu_ms"] > 0 and st["d2h_bytes"] >= len(runs[2][1]) and st["arena_nodes"] > 1_000_000


@pytest.mark.gpu
def test_stats_extend_the_root_entry(ctx):
    keys, off, vals = shuffled_sorted_leaves(50_000, seed=41)
    ctx.trie_root_leaves(keys, off, vals)
    want = ctx.stats()
    _, got_bytes = ctx.trie_subset_leaves(keys, off, vals, keys[:1000])
    got = ctx.stats()
    for f in ("nodes_hashed", "node_permutations", "node_bytes", "arena_nodes", "levels"):
        assert got[f] == want[f], f
    assert got["kernel_launches"] > want["kernel_launches"]
    assert got["d2h_bytes"] >= want["d2h_bytes"] + len(got_bytes)


# ---------------------------------------------------------------- round trip through the witness parser -------------
EMPTY_CODE_HASH = bytes.fromhex("c5d2460186f7233c927e7db2dcc703c0e500b653ca82273b7bfad8045d85a470")


def account_template():
    """rlp([nonce (8 bytes), balance (16 bytes), EMPTY_TRIE_ROOT, keccak("")]) with nonce at [3, 11), balance at [12, 28)"""
    from proof_protocol_decoder_b200 import synth

    t = synth.rlp_list([synth.rlp_str(b"\x01" * 8), synth.rlp_str(b"\x01" * 16), synth.rlp_str(tm.EMPTY_TRIE_HASH), synth.rlp_str(EMPTY_CODE_HASH)])
    assert len(t) == 94 and t[2] == 0x88 and t[11] == 0x90
    return np.frombuffer(t, dtype=np.uint8)


def _round_trip(ctx, lib, root, subset):
    from proof_protocol_decoder_b200 import flat

    witness = lib.direct_to_compact(flat.encode_direct_pre_image(subset, {}))
    assert flat.parse_pre_image_dump(ctx.compact_decode(witness))["state_root"] == root


@pytest.mark.gpu
def test_round_trip_one_million_accounts(ctx):
    from proof_protocol_decoder_b200 import synth

    rng = np.random.default_rng(43)
    n = 1_000_000
    keys = synth.gen_sorted_leaves(n, seed=43)[0]
    vals = np.tile(account_template(), (n, 1))
    vals[:, 3:11] = np.frombuffer(rng.bytes(8 * n), dtype=np.uint8).reshape(n, 8) | np.array([1] + [0] * 7, np.uint8)
    vals[:, 12:28] = np.frombuffer(rng.bytes(16 * n), dtype=np.uint8).reshape(n, 16) | np.array([1] + [0] * 15, np.uint8)
    off = np.arange(n + 1, dtype=np.uint64) * 94
    vals = vals.reshape(-1)
    keys, off, vals = permute(keys, off, vals, rng.permutation(n))
    root, subset = ctx.trie_subset_leaves(keys, off, vals, mixed_queries(keys, 100_000, rng))
    assert root == ctx.trie_root_leaves(keys, off, vals)
    _round_trip(ctx, ctx.lib, root, subset)


@pytest.mark.gpu
def test_round_trip_ten_million_device_accounts(ctx):
    import torch

    from proof_protocol_decoder_b200 import synth

    n, m = 10_000_000, 100_000
    keys, _, _ = synth.gen_sorted_leaves_dev(n, seed=47)
    g = torch.Generator(device="cuda")
    g.manual_seed(47)
    vals = torch.from_numpy(account_template().copy()).cuda().repeat(n, 1)
    lead = torch.zeros(8, dtype=torch.uint8, device="cuda")
    lead[0] = 1
    vals[:, 3:11] = torch.randint(0, 256, (n, 8), dtype=torch.uint8, device="cuda", generator=g) | lead
    vals[:, 12:28] = torch.randint(0, 256, (n, 16), dtype=torch.uint8, device="cuda", generator=g) | torch.cat([lead, torch.zeros(8, dtype=torch.uint8, device="cuda")])
    vals = vals.reshape(-1)
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * 94
    pick = torch.randint(0, n, (m // 2,), device="cuda", generator=g)
    q = torch.cat([keys[pick], torch.randint(0, 256, (m - m // 2, 32), dtype=torch.uint8, device="cuda", generator=g)])
    torch.cuda.synchronize()
    want = ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel())
    root, subset = ctx.trie_subset_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel(), q.data_ptr(), m)
    assert root == want
    assert ctx.trie_subset_leaves_dev(keys.data_ptr(), 32, off.data_ptr(), vals.data_ptr(), n, vals.numel(), q.data_ptr(), m) == (root, subset)
    _round_trip(ctx, ctx.lib, root, subset)
