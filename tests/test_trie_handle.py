"""Resident trie handles (ppd_trie_*): a trie built once from leaves, cut into subsets and updated in place.

CPU: a dict model (the surviving items, sorted, through trie_model) against the oracle's insert / delete sequence
(tests/cpp/trie_update_oracle.cpp).  GPU: chains of update batches against the oracle, the model and the one-shot root
and subset entries on the numpy-merged leaves; incrementality (nodes_hashed), hashed keys, argument errors that leave
the handle as it was, and a context shared with one-shot calls and other handles."""
import ctypes

import numpy as np
import pytest

import trie_model as tm
from test_node_encoding_edges import _arrays, _bytes_key, gadgets, union
from test_trie_subset import mixed_queries, probes, structured_set
from test_unsorted_leaves import _dev, pack, rand_values, shuffled_sorted_leaves

BAD_ARGUMENT = 62
EMPTY_TRIE_HASH = bytes.fromhex("56e81f171bcc55a6ff8345e692c0f86e5b48e01b996cadc001622fb5e363b421")


@pytest.fixture(scope="module")
def ctx():
    from proof_protocol_decoder_b200.lib import Context

    c = Context(0)
    yield c
    c.close()


class UpdateOracle:
    def __init__(self, so_path):
        self.L = ctypes.CDLL(str(so_path))
        vp, sz = ctypes.c_void_p, ctypes.c_size_t
        u8p = ctypes.POINTER(ctypes.c_uint8)
        self.L.oracle_trie_update.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp, sz, vp, sz, ctypes.c_char_p, ctypes.POINTER(u8p), ctypes.POINTER(sz),
                                              ctypes.c_char_p, sz]
        self.L.oracle_free.argtypes = [vp]

    def run(self, leaves, batches, queries=None):
        """root (and subset for the queries) after inserting the leaves, then every (keys, del, off, vals) batch in order"""
        keys, off, vals = (np.ascontiguousarray(a) for a in leaves)
        uk = np.concatenate([b[0] for b in batches]) if batches else np.zeros((0, 32), np.uint8)
        ud = np.concatenate([b[1] for b in batches]).astype(np.uint8) if batches else np.zeros(0, np.uint8)
        uv = [v for b in batches for v in values_of(b[2], b[3])]
        uo, uvals = pack(uv) if uv else (np.zeros(1, np.uint64), np.zeros(1, np.uint8))
        root = ctypes.create_string_buffer(32)
        out, n = ctypes.POINTER(ctypes.c_uint8)(), ctypes.c_size_t()
        err = ctypes.create_string_buffer(512)
        q = np.ascontiguousarray(queries if queries is not None else np.zeros((0, 32), np.uint8), dtype=np.uint8)
        rc = self.L.oracle_trie_update(keys.ctypes.data, off.ctypes.data, vals.ctypes.data, len(keys), np.ascontiguousarray(uk).ctypes.data,
                                       ud.ctypes.data, uo.ctypes.data, uvals.ctypes.data, len(uk), q.ctypes.data, len(q), root,
                                       ctypes.byref(out) if queries is not None else None, ctypes.byref(n), err, 512)
        assert rc == 0, err.value
        if queries is None:
            return root.raw
        sub = ctypes.string_at(out, n.value)
        self.L.oracle_free(out)
        return root.raw, sub


@pytest.fixture(scope="module")
def update_oracle(tmp_path_factory):
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    so = tmp_path_factory.mktemp("update_oracle") / "libtrie_update_oracle.so"
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", str(so), os.path.join(root, "tests", "cpp", "trie_update_oracle.cpp")])
    return UpdateOracle(so)


def values_of(off, vals):
    return [bytes(vals[int(off[i]) : int(off[i + 1])]) for i in range(len(off) - 1)]


# ---------------------------------------------------------------- the model ------------------------------------------
def apply(state, batch):
    keys, dels, off, vals = batch
    for k, d, v in zip(keys, dels, values_of(off, vals)):
        if d:
            state.pop(bytes(k), None)
        else:
            state[bytes(k)] = v
    return state


def model_root(state):
    if not state:
        return EMPTY_TRIE_HASH
    items = [(tm.nibbles(k), state[k]) for k in sorted(state)]
    return tm.keccak(tm.node_rlp(items, 0))


def state_arrays(state):
    ks = sorted(state)
    keys = np.frombuffer(b"".join(ks), dtype=np.uint8).reshape(-1, 32).copy() if ks else np.zeros((0, 32), np.uint8)
    off, vals = pack([state[k] for k in ks]) if ks else (np.zeros(1, np.uint64), np.zeros(1, np.uint8))
    return keys, off, vals


def make_batch(rng, present, k, frac=(0.6, 0.3, 0.1)):
    """k updates in any order: overwrites of present keys, new keys, deletes of present keys"""
    n_ow = int(k * frac[0]) if len(present) else 0
    n_del = int(k * frac[2]) if len(present) else 0
    n_new = k - n_ow - n_del
    ow = present[rng.integers(0, len(present), size=n_ow)] if n_ow else np.zeros((0, 32), np.uint8)
    de = present[rng.integers(0, len(present), size=n_del)] if n_del else np.zeros((0, 32), np.uint8)
    new = np.frombuffer(rng.bytes(32 * n_new), dtype=np.uint8).reshape(-1, 32)
    keys = np.concatenate([ow, new, de])
    dels = np.concatenate([np.zeros(n_ow + n_new, np.uint8), np.ones(n_del, np.uint8)])
    perm = rng.permutation(len(keys))
    keys, dels = np.ascontiguousarray(keys[perm]), dels[perm]
    off, vals = pack([b"" if d else v for d, v in zip(dels, rand_values(rng, len(keys), 1, 40))])
    return keys, dels, off, vals


# ---------------------------------------------------------------- CPU: the model against the oracle ------------------
@pytest.mark.parametrize("seed", [1, 2])
def test_model_equals_oracle_random_batches(update_oracle, seed):
    rng = np.random.default_rng(seed)
    keys, off, vals = structured_set(rng, 300)
    state = dict(zip(map(bytes, keys), values_of(off, vals)))
    batches = []
    for _ in range(4):
        b = make_batch(rng, state_arrays(state)[0], 60)
        batches.append(b)
        apply(state, b)
        assert update_oracle.run((keys, off, vals), batches) == model_root(state)


def test_model_equals_oracle_deletes_collapse_every_gadget(update_oracle):
    items = union("raw")
    keys, off, vals = _arrays(items)
    state = dict(zip(map(bytes, keys), values_of(off, vals)))
    for name, its in gadgets("raw"):
        gk = np.array([list(_bytes_key(k)) for k, _ in its], dtype=np.uint8)
        for r in range(len(gk)):  # delete one key of the gadget: its branch or extension collapses
            b = (gk[r : r + 1], np.ones(1, np.uint8), *pack([b""]))
            s = apply(dict(state), b)
            assert update_oracle.run((keys, off, vals), [b]) == model_root(s), name


def test_model_equals_oracle_absent_rewrite_and_delete_all(update_oracle):
    rng = np.random.default_rng(7)
    keys, off, vals = structured_set(rng, 100)
    state = dict(zip(map(bytes, keys), values_of(off, vals)))
    absent = probes(keys, rng, 2)
    b1 = (absent, np.ones(len(absent), np.uint8), *pack([b""] * len(absent)))  # deletes of absent keys: nothing changes
    assert update_oracle.run((keys, off, vals), [b1]) == model_root(state)
    k0 = keys[:3]
    b2 = (np.concatenate([k0, k0]), np.array([1, 1, 1, 0, 0, 0], np.uint8), *pack([b""] * 3 + [b"\x05", b"\x06", b"\x07"]))  # delete, then write
    b3 = (np.concatenate([k0, k0]), np.array([0, 0, 0, 1, 1, 1], np.uint8), *pack([b"\x05", b"\x06", b"\x07"] + [b""] * 3))  # write, then delete
    for b in (b2, b3):
        assert update_oracle.run((keys, off, vals), [b]) == model_root(apply(dict(state), b))
    ball = (keys, np.ones(len(keys), np.uint8), *pack([b""] * len(keys)))
    assert update_oracle.run((keys, off, vals), [ball]) == EMPTY_TRIE_HASH == model_root({})


# ---------------------------------------------------------------- GPU -------------------------------------------------
def _check_handle(ctx, t, state, queries, oracle=None, leaves=None, batches=None):
    keys, off, vals = state_arrays(state)
    want = ctx.trie_root_leaves(keys, off, vals)
    assert t.root == want and t.n == len(keys)
    if len(keys) <= 10_000:
        assert t.root == model_root(state)
    if oracle is not None:
        oroot, osub = oracle.run(leaves, batches, queries)
        assert t.root == oroot
        assert t.subset(queries) == osub
    root, sub = ctx.trie_subset_leaves(keys, off, vals, queries)
    assert root == t.root
    assert t.subset(queries) == sub, "handle subset vs the one-shot subset on the merged leaves"


@pytest.mark.gpu
@pytest.mark.parametrize("n", [0, 1, 2, 1000, 100_000, 1_000_000])
def test_update_chains(ctx, update_oracle, n):
    rng = np.random.default_rng(n + 11)
    if n:
        keys, off, vals = shuffled_sorted_leaves(n, seed=n + 5)
    else:
        keys, off, vals = np.zeros((0, 32), np.uint8), np.zeros(1, np.uint64), np.zeros(1, np.uint8)
    state = dict(zip(map(bytes, keys), values_of(off, vals))) if n <= 100_000 else None
    with ctx.trie_from_leaves(keys, off, vals) as t:
        assert t.root == ctx.trie_root_leaves(keys, off, vals)
        batches = []
        cur = (keys, off, vals)
        for step in range(6):
            present = state_arrays(state)[0] if state is not None else cur[0]
            k = [1, 10, 100, 1000, 3, 500][step] if n < 1_000_000 else [1000, 10_000, 100_000, 1, 5000, 20_000][step]
            b = make_batch(rng, present, k)
            batches.append(b)
            got = t.update(b[0], b[2], b[3], deletes=b[1])
            if state is not None:
                apply(state, b)
                small = n <= 1000
                _check_handle(ctx, t, state, mixed_queries(state_arrays(state)[0], 200, rng), update_oracle if small else None, (keys, off, vals), batches)
            else:
                cur = merge_np(cur, b)
                assert got == ctx.trie_root_leaves(*cur)
                q = mixed_queries(cur[0], 1000, rng)
                assert t.subset(q) == ctx.trie_subset_leaves(*cur, q)[1]


def merge_np(cur, batch):
    """numpy merge of sorted leaves and a batch (last update of a key wins; deletes drop)"""
    keys, off, vals = cur
    uk, ud, uo, uv = batch
    allk = np.concatenate([keys, uk]).view("S32").ravel()
    n = len(allk)
    rev = allk[::-1]
    _, idx = np.unique(rev, return_index=True)
    last = n - 1 - idx
    isdel = np.concatenate([np.zeros(len(keys), np.uint8), ud])[last].astype(bool)
    last = last[~isdel]
    ov, nv = values_of(off, vals), values_of(uo, uv)
    allv = ov + nv
    nk = np.concatenate([keys, uk])[last]
    if len(nk) == 0:
        return np.zeros((0, 32), np.uint8), np.zeros(1, np.uint64), np.zeros(1, np.uint8)
    o, v = pack([allv[i] for i in last])
    return np.ascontiguousarray(nk), o, v


@pytest.mark.gpu
def test_gadgets_delete_one_by_one_then_reinsert(ctx):
    items = union("raw")
    keys, off, vals = _arrays(items)
    state = dict(zip(map(bytes, keys), values_of(off, vals)))
    rng = np.random.default_rng(3)
    with ctx.trie_from_leaves(keys, off, vals) as t:
        for r in range(len(keys)):
            b = (keys[r : r + 1], np.ones(1, np.uint8), *pack([b""]))
            t.update(b[0], b[2], b[3], deletes=b[1])
            apply(state, b)
            assert t.root == model_root(state)
            if r % 16 == 0:
                _check_handle(ctx, t, state, mixed_queries(keys, 40, rng))
        assert t.root == EMPTY_TRIE_HASH and t.n == 0
        assert t.subset(keys[:3]) == bytes([0])
        for r in range(len(keys)):
            v = values_of(off, vals)[r]
            b = (keys[r : r + 1], np.zeros(1, np.uint8), *pack([v]))
            t.update(b[0], b[2], b[3], deletes=b[1])
            apply(state, b)
            assert t.root == model_root(state)
        _check_handle(ctx, t, state, np.concatenate([keys, probes(keys, rng, 4)]))


@pytest.mark.gpu
def test_updates_rehash_only_changed_paths(ctx):
    rng = np.random.default_rng(5)
    keys, off, vals = shuffled_sorted_leaves(1_000_000, seed=9)
    root = ctx.trie_root_leaves(keys, off, vals)
    assert ctx.stats()["nodes_hashed"] > 1_000_000
    with ctx.trie_from_leaves(keys, off, vals) as t:
        assert t.root == root
        cur = (keys, off, vals)
        b = make_batch(rng, keys, 1, (1.0, 0, 0))
        t.update(b[0], b[2], b[3], deletes=b[1])
        assert ctx.stats()["nodes_hashed"] <= 32
        cur = merge_np(cur, b)
        assert t.root == ctx.trie_root_leaves(*cur)
        b = make_batch(rng, keys, 1000)
        t.update(b[0], b[2], b[3], deletes=b[1])
        assert ctx.stats()["nodes_hashed"] <= 32_000
        cur = merge_np(cur, b)
        assert t.root == ctx.trie_root_leaves(*cur)
        before = t.root
        assert t.update(np.zeros((0, 32), np.uint8), np.zeros(1, np.uint64), np.zeros(1, np.uint8)) == before
        assert ctx.stats()["nodes_hashed"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("key_len", [20, 32])
def test_hashed_keys(ctx, key_len):
    rng = np.random.default_rng(key_len)
    raw = np.frombuffer(rng.bytes(key_len * 3000), dtype=np.uint8).reshape(-1, key_len)
    off, vals = pack(rand_values(rng, len(raw)))
    with ctx.trie_from_leaves(raw, off, vals, hash_keys=True) as t:
        assert t.root == ctx.trie_root_leaves(raw, off, vals, hash_keys=True)
        newk = np.frombuffer(rng.bytes(key_len * 200), dtype=np.uint8).reshape(-1, key_len)
        uk = np.concatenate([raw[:300], newk])
        dels = np.concatenate([np.ones(100, np.uint8), np.zeros(400, np.uint8)])
        uo, uv = pack([b"" if d else v for d, v in zip(dels, rand_values(rng, len(uk)))])
        t.update(uk, uo, uv, deletes=dels)
        # the same leaves, in insertion order, through the one-shot entry: deleted keys simply left out
        keep = np.ones(len(raw), bool)
        keep[:100] = False
        allk = np.concatenate([raw[keep], uk[100:]])
        av = [v for i, v in enumerate(values_of(off, vals)) if keep[i]] + values_of(uo, uv)[100:]
        ao, avals = pack(av)
        assert t.root == ctx.trie_root_leaves(allk, ao, avals, hash_keys=True)
        q = np.concatenate([raw[:50], newk[:50]])
        assert t.subset(q) == ctx.trie_subset_leaves(allk, ao, avals, q, hash_keys=True)[1]


@pytest.mark.gpu
def test_errors_leave_the_handle_unchanged(ctx):
    import torch

    from proof_protocol_decoder_b200.lib import PpdError

    rng = np.random.default_rng(8)
    keys, off, vals = shuffled_sorted_leaves(5000, seed=4)
    q = mixed_queries(keys, 300, rng)
    with ctx.trie_from_leaves(keys, off, vals) as t:
        root, sub = t.root, t.subset(q)
        b = make_batch(rng, keys, 100)
        bad_off = b[2].copy()
        bad_off[50] = bad_off[51] + 1  # decreasing
        dk, do, dv = _dev(b[0], bad_off, b[3])
        torch.cuda.synchronize()
        with pytest.raises(PpdError) as e:
            t.update_dev(dk.data_ptr(), None, do.data_ptr(), dv.data_ptr(), 100, dv.numel())
        assert e.value.code == BAD_ARGUMENT
        with pytest.raises(PpdError) as e:
            t.update_dev(dk.data_ptr(), None, do.data_ptr(), dv.data_ptr(), 2**31 - 2, dv.numel())
        assert e.value.code == BAD_ARGUMENT
        other = type(ctx)(0)
        try:
            r = ctypes.create_string_buffer(32)
            assert other.lib.L.ppd_trie_update_dev(other.h, t.h, dk.data_ptr(), None, do.data_ptr(), dv.data_ptr(), 100, dv.numel(), r) == BAD_ARGUMENT
        finally:
            other.close()
        assert ctx.lib.L.ppd_trie_update_dev(ctx.h, None, dk.data_ptr(), None, do.data_ptr(), dv.data_ptr(), 100, dv.numel(), r) == BAD_ARGUMENT
        assert t.root == root and t.subset(q) == sub and t.n == 5000
        t.update(b[0], b[2], b[3], deletes=b[1])
        assert t.root == ctx.trie_root_leaves(*merge_np((keys, off, vals), b))


@pytest.mark.gpu
def test_mixed_use_of_one_context_and_lifetime(ctx):
    import os
    import sys

    import torch

    from proof_protocol_decoder_b200 import synth
    from proof_protocol_decoder_b200.lib import Context

    rng = np.random.default_rng(12)
    a = shuffled_sorted_leaves(20_000, seed=21)
    b = shuffled_sorted_leaves(30_000, seed=22)
    ta, tb = ctx.trie_from_leaves(*a), ctx.trie_from_leaves(*b)
    ca, cb = a, b
    blk = synth.gen_block(7, n_accounts=200, n_txns=4, n_withdrawals=1)
    for step in range(3):
        ba, bb = make_batch(rng, ca[0], 300), make_batch(rng, cb[0], 700)
        ta.update(ba[0], ba[2], ba[3], deletes=ba[1])
        ca = merge_np(ca, ba)
        ctx.trie_root_leaves(*shuffled_sorted_leaves(40_000, seed=step))  # one-shot calls reuse the context's scratch
        ctx.trie_subset_leaves(*b, b[0][:10])
        ctx.block_decode(blk.flat)
        tb.update(bb[0], bb[2], bb[3], deletes=bb[1])
        cb = merge_np(cb, bb)
        for t, cur in ((ta, ca), (tb, cb)):
            q = mixed_queries(cur[0], 100, rng)
            assert t.root == ctx.trie_root_leaves(*cur)
            assert t.subset(q) == ctx.trie_subset_leaves(*cur, q)[1]
    # host and device entries agree, inputs are not modified
    keys, off, vals = shuffled_sorted_leaves(3000, seed=31)
    dk, do, dv = _dev(keys, off, vals)
    sk = np.ascontiguousarray(keys[np.lexsort(keys.T[::-1])])
    torch.cuda.synchronize()
    with ctx.trie_from_leaves_dev(dk.data_ptr(), 32, do.data_ptr(), dv.data_ptr(), len(keys), dv.numel()) as td, ctx.trie_from_leaves(keys, off, vals) as th:
        assert td.root == th.root == ctx.trie_root_leaves(keys, off, vals)
        bt = make_batch(rng, keys, 200)
        ek, eo, ev = _dev(bt[0], bt[2], bt[3])
        ed = torch.from_numpy(bt[1]).cuda()
        torch.cuda.synchronize()
        copies = [x.clone() for x in (dk, do, dv, ek, eo, ev, ed)]
        assert td.update_dev(ek.data_ptr(), ed.data_ptr(), eo.data_ptr(), ev.data_ptr(), len(bt[0]), ev.numel()) == th.update(bt[0], bt[2], bt[3], deletes=bt[1])
        q = mixed_queries(keys, 100, rng)
        qd = torch.from_numpy(q).cuda()
        torch.cuda.synchronize()
        assert td.subset_dev(qd.data_ptr(), len(q)) == th.subset(q)
        for x, y in zip((dk, do, dv, ek, eo, ev, ed), copies):
            assert torch.equal(x, y)
    del sk
    # a context destroyed with live handles releases them
    c2 = Context(0)
    t2 = c2.trie_from_leaves(*a)
    t3 = c2.trie_from_leaves(*b)
    assert t2.root == ctx.trie_root_leaves(*a) and t3.n == len(b[0])
    c2.close()
    t2.close()  # the context took it: a no-op
    ta.close(), tb.close()


@pytest.mark.gpu
def test_sorted_create_and_round_trip_ten_million(ctx):
    import torch

    from proof_protocol_decoder_b200 import synth
    from test_trie_subset import _round_trip, account_template

    n = 10_000_000
    keys, _, _ = synth.gen_sorted_leaves_dev(n, seed=77)
    vals = torch.from_numpy(account_template().copy()).cuda().repeat(n, 1).reshape(-1)
    off = torch.arange(n + 1, dtype=torch.int64, device="cuda") * 94
    torch.cuda.synchronize()
    want = ctx.trie_root_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel())
    rng = np.random.default_rng(4)
    acct = account_template().tobytes()
    with ctx.trie_from_sorted_leaves_dev(keys.data_ptr(), off.data_ptr(), vals.data_ptr(), n, vals.numel()) as t:
        assert t.root == want and t.n == n
        present = keys[torch.from_numpy(rng.integers(0, n, size=20_000)).cuda()].cpu().numpy()
        for _ in range(3):
            b = make_batch(rng, present, 10_000)
            uo, uv = pack([b"" if d else acct[:3] + bytes([1 + int(rng.integers(0, 255))]) + rng.bytes(7) + acct[11:] for d in b[1]])
            t.update(b[0], uo, uv, deletes=b[1])
        q = np.concatenate([present[:1000], b[0][:1000], mixed_queries(present, 1000, rng)])
        sub = t.subset(q)
        _round_trip(ctx, ctx.lib, t.root, sub)


# ---------------------------------------------------------------- collapses at every depth, growth, alignment ---------
def collapse_sets(rng):
    """for every depth d: a pair of keys under a branch at depth d with only those two children (plus, from d = 1 on, a
    key that leaves at nibble 0, so that an extension leads down to the pair's branch from d = 2 on)"""
    out = []
    for d in range(64):
        p = tm.nibbles(rng.bytes(32))
        a, b = list(p), list(p)
        b[d] = (a[d] + 1 + int(rng.integers(0, 15))) % 16
        keys = [a, b]
        if d:
            c = tm.nibbles(rng.bytes(32))
            c[0] = (a[0] + 1) % 16
            keys.append(c)
        k = np.array([list(_bytes_key(x)) for x in keys], dtype=np.uint8)
        off, vals = pack(rand_values(rng, len(k), 1, 40))
        out.append((d, k, off, vals))
    return out


def test_model_equals_oracle_collapse_at_every_depth(update_oracle):
    rng = np.random.default_rng(17)
    for d, keys, off, vals in collapse_sets(rng):
        for r in (0, 1):  # delete either key of the pair: the branch at depth d collapses into the other's leaf
            b = (keys[r : r + 1], np.ones(1, np.uint8), *pack([b""]))
            s = apply(dict(zip(map(bytes, keys), values_of(off, vals))), b)
            assert update_oracle.run((keys, off, vals), [b]) == model_root(s), d


@pytest.mark.gpu
def test_collapse_at_every_depth(ctx):
    rng = np.random.default_rng(17)
    for d, keys, off, vals in collapse_sets(rng):
        for r in (0, 1):
            state = dict(zip(map(bytes, keys), values_of(off, vals)))
            with ctx.trie_from_leaves(keys, off, vals) as t:
                b = (keys[r : r + 1], np.ones(1, np.uint8), *pack([b""]))
                t.update(b[0], b[2], b[3], deletes=b[1])
                apply(state, b)
                assert t.root == model_root(state), d
                _check_handle(ctx, t, state, np.concatenate([keys, probes(keys, rng, 1)]))
                b = (keys[r : r + 1], np.zeros(1, np.uint8), *pack([values_of(off, vals)[r]]))  # and back
                t.update(b[0], b[2], b[3], deletes=b[1])
                apply(state, b)
                assert t.root == model_root(state) == ctx.trie_root_leaves(keys, off, vals), d


@pytest.mark.gpu
def test_batches_that_grow_the_trie_several_times(ctx):
    """batches of new keys that double and triple the trie: the merge's scratch follows the new size"""
    rng = np.random.default_rng(23)
    cur = shuffled_sorted_leaves(100_000, seed=41)
    with ctx.trie_from_leaves(*cur) as t:
        for k in (150_000, 500_000):
            b = make_batch(rng, cur[0], k, (0.0, 1.0, 0.0))
            t.update(b[0], b[2], b[3], deletes=b[1])
            cur = merge_np(cur, b)
            assert t.n == len(cur[0]) and t.root == ctx.trie_root_leaves(*cur)
            q = mixed_queries(cur[0], 2000, rng)
            assert t.subset(q) == ctx.trie_subset_leaves(*cur, q)[1]
    one = shuffled_sorted_leaves(1_000_000, seed=42)
    with ctx.trie_from_leaves(*one) as t:  # in a fresh handle: 1 M new keys on 1 M leaves
        b = make_batch(rng, one[0], 1_000_000, (0.0, 1.0, 0.0))
        t.update(b[0], b[2], b[3], deletes=b[1])
        assert t.n == 2_000_000 and t.root == ctx.trie_root_leaves(*merge_np(one, b))


@pytest.mark.gpu
def test_unaligned_device_keys_values_and_queries(ctx):
    import torch

    rng = np.random.default_rng(29)
    leaves = shuffled_sorted_leaves(20_000, seed=43)
    b = make_batch(rng, leaves[0], 3000)
    q = mixed_queries(leaves[0], 500, rng)

    def at(arr, shift):  # a device copy of arr that starts `shift` bytes into its allocation
        flat = np.ascontiguousarray(arr, dtype=np.uint8).reshape(-1)
        buf = torch.zeros(flat.size + 16, dtype=torch.uint8, device="cuda")
        buf[shift : shift + flat.size] = torch.from_numpy(flat).cuda()
        return buf, buf.data_ptr() + shift

    with ctx.trie_from_leaves(*leaves) as ta, ctx.trie_from_leaves(*leaves) as tu:
        ka, _ = at(b[0], 0)
        ku, pku = at(b[0], 1)
        va, _ = at(b[3], 0)
        vu, pvu = at(b[3], 3)
        da, _ = at(b[1], 0)
        du, pdu = at(b[1], 5)
        o = torch.from_numpy(b[2].astype(np.int64)).cuda()
        torch.cuda.synchronize()
        want = ta.update_dev(ka.data_ptr(), da.data_ptr(), o.data_ptr(), va.data_ptr(), len(b[0]), b[3].size)
        assert tu.update_dev(pku, pdu, o.data_ptr(), pvu, len(b[0]), b[3].size) == want
        assert want == ctx.trie_root_leaves(*merge_np(leaves, b))
        qa, _ = at(q, 0)
        qu, pqu = at(q, 1)
        torch.cuda.synchronize()
        assert tu.subset_dev(pqu, len(q)) == ta.subset_dev(qa.data_ptr(), len(q)) == ta.subset(q)


@pytest.mark.gpu
def test_sorted_create_checks_offsets_against_vals_bytes(ctx):
    import torch

    from proof_protocol_decoder_b200.lib import PpdError

    keys, off, vals = shuffled_sorted_leaves(1000, seed=44)
    sk = np.ascontiguousarray(keys[np.lexsort(keys.T[::-1])])
    k, o, v = _dev(sk, off, vals)
    torch.cuda.synchronize()
    with pytest.raises(PpdError) as e:
        ctx.trie_from_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), len(sk), int(off[-1]) - 1)
    assert e.value.code == BAD_ARGUMENT
    with ctx.trie_from_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), len(sk), int(off[-1])) as t:
        assert t.root == ctx.trie_root_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), len(sk), int(off[-1]))
