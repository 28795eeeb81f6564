"""Both CUDA trie hashers at every node-encoding boundary, against the recursive model (trie_model.py) and the oracle.

The two encoders (the sorted-leaves builder of ppd_build.cu and the arena level hasher of ppd_kernels.cu) emit RLP into a
per-thread Keccak stage; their risky decisions sit on byte counts: inline or hashed (< 32), 1 / 2 / 3 list-header bytes
(56, 256, 65 536), the single-byte string rule (< 0x80), the number of 136-byte rate blocks (filled in 128-byte value
units or three-child branch units) and the nibble shift of odd key starts.  Random tries hit these only by chance.

The cases here are built to land on them.  A gadget is a few sorted (key, value) items under its own two-nibble prefix;
where a node must encode to an exact length, a value length is found by searching with the model.  The coverage tests
walk the model's nodes and fail when a boundary is no longer reached, so a change of the generator cannot drift off
them silently.

Two forms of the same gadgets: "raw", values as the sorted-leaves API takes them (the trie value itself), and
"witness", storage tries of a compact witness, whose trie value is rlp_str(witness value)."""
import functools
import os

import numpy as np
import pytest

import trie_model as tm
import witness_shapes as ws
from proof_protocol_decoder_b200 import synth

EMPTY_CODE_HASH = synth.keccak256(b"")
FORMS = {"raw": lambda w: w, "witness": synth.rlp_str}

# ---------------------------------------------------------------- targets -------------------------------------------
LEAF_NIBBLES = {0, 1, 2, 3, 55, 62, 63}
LEAF_TOTALS = {31, 32, 135, 136, 137, 271, 272, 273}
LIST_PAYLOADS = {55, 56, 255, 256}
VALUE_LENGTHS = {0, 1, 55, 56, 127, 128, 129, 255, 256, 65535, 65536}
ONE_BYTE_VALUES = {0x00, 0x7F, 0x80, 0xFF}
BRANCH_TOTALS = {31, 32, 135, 136, 137, 271, 272, 273, 407, 408, 409}
BRANCH_PAYLOADS = {255, 256}
EXT_NIBBLES = [1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 17, 58]
EXT_TOTALS = {31, 32}


def _list_len(payload):
    return payload + (1 if payload < 56 else 2 if payload < 256 else 3)


def _val(n, seed=0):
    return bytes((seed * 29 + 37 * i + 1) & 255 for i in range(n))


def _key(head, seed=0):
    """the nibbles `head`, then a fixed pattern up to 64 nibbles"""
    return list(head) + [(seed * 7 + 3 * i + 1) % 16 for i in range(64 - len(head))]


def _fill(pfx, depth, seed=0):
    """pfx extended to `depth` nibbles"""
    return _key(pfx, seed)[:depth]


def _model_items(items_w, form):
    return sorted((k, FORMS[form](w)) for k, w in items_w)


def _node_len(items_w, form, kind, depth):
    """the encoded length of the node at `depth` above items_w[0] if it is of `kind` (the model, on that subtree only)"""
    key = items_w[0][0]
    sub = _model_items([it for it in items_w if it[0][:depth] == key[:depth]], form)
    is_kind = "leaf" if len(sub) == 1 else "ext" if tm.common_depth(sub, depth) > depth else "branch"
    return len(tm.node_rlp(sub, depth)) if is_kind == kind else None


def _tune(make, form, kind, depth, target, ns):
    """make(n) for the first n for which the node at `depth` above the first item encodes to `target` bytes"""
    for n in ns:
        items = make(n)
        if _node_len(items, form, kind, depth) == target:
            return items
    return None


# ---------------------------------------------------------------- gadgets -------------------------------------------
def _leaf_pair(pfx, r, w_a, w_b=b"\x01"):
    """two leaves with r key nibbles left, below a branch at depth 63 - r (r <= 61)"""
    base = _fill(pfx, 63 - r, r)
    return [(base + [3] + _key([], 1)[:r], w_a), (base + [9] + _key([], 2)[:r], w_b)]


def _branch(pfx, depth, slots, values):
    """a branch at `depth` whose children are leaves; values[j] is the value of the j-th child"""
    base = _fill(pfx, depth, depth)
    return [(base + [s] + _key([], s)[: 63 - depth], values[j]) for j, s in enumerate(slots)]


def _ext(pfx, s, e, kid_values, parity_seed=0):
    """an extension of e nibbles at depth s (below a branch at s - 1 that also holds a filler leaf) over a branch at
    depth s + e with two leaf children"""
    base = _fill(pfx, s - 1, parity_seed)
    mid = base + [4] + _key([], 5 + parity_seed)[:e]
    r = 63 - (s + e)
    kids = [(mid + [c] + _key([], c)[:r], w) for c, w in zip((2, 13), kid_values)]
    return kids + [(base + [11] + _key([], 11)[: 64 - s], _val(20, 3))]


def _leaf_gadgets(form):
    out = []
    rs = [0, 1, 2, 3, 7, 30, 55]
    k = 0
    for n in sorted(VALUE_LENGTHS):
        firsts = sorted(ONE_BYTE_VALUES) if n == 1 else [0x42]
        for f in firsts:
            w = bytes([f]) + _val(n - 1, n) if n else b""
            out.append((f"leaf_value_{n}_{f:02x}", lambda p, w=w, r=rs[k % len(rs)]: _leaf_pair(p, r, w)))
            k += 1
    for t in sorted(LEAF_TOTALS):
        out.append((f"leaf_total_{t}", functools.partial(_tuned_leaf, form=form, total=t)))
    for pl in sorted(LIST_PAYLOADS):
        out.append((f"leaf_payload_{pl}", functools.partial(_tuned_leaf, form=form, total=_list_len(pl))))
    return out


def _tuned_leaf(pfx, form, total):
    for r in (0, 1, 3, 2, 55, 20, 61):
        items = _tune(lambda n: _leaf_pair(pfx, r, _val(n, total)), form, "leaf", 64 - r, total, range(1, 400))
        if items:
            return items
    raise AssertionError(f"no leaf of {total} bytes")


def _branch_gadgets(form):
    small = b"\x01"
    out = []
    for k in range(2, 17):
        # children alternately inline and hashed: slot 0 present in the first form, slot 15 in the second
        for name, slots, inl in (("low", list(range(k)), 0), ("high", list(range(16 - k, 16)), 1)):
            vals = [small if (j + inl) % 2 == 0 else _val(40, j) for j in range(k)]
            out.append((f"branch_{k}_{name}", lambda p, s=slots, v=vals: _branch(p, 60, s, v)))
    out.append(("branch_16_inline", lambda p: _branch(p, 60, list(range(16)), [small] * 16)))
    out.append(("branch_3_spread", lambda p: _branch(p, 60, [1, 8, 14], [small, _val(40), small])))
    for t in sorted(BRANCH_TOTALS) + [_list_len(pl) for pl in sorted(BRANCH_PAYLOADS)]:
        out.append((f"branch_total_{t}", functools.partial(_tuned_branch, form=form, total=t)))
    return out


def _tuned_branch(pfx, form, total):
    depth = 60 if total > 32 else 62
    for k in range(2, 17):
        slots = list(range(0, 16, 16 // k))[:k] if k <= 8 else list(range(k))
        for h in range(k - 1, -1, -1):
            def make(n):
                vals = [_val(n, total)] + [b"\x01"] * (k - h - 1) + [_val(40, j) for j in range(h)]
                return _branch(pfx, depth, slots, vals)

            items = _tune(make, form, "branch", depth, total, range(1, 30))
            if items:
                return items
    raise AssertionError(f"no branch of {total} bytes")


def _ext_gadgets(form):
    out = []
    for e in EXT_NIBBLES:
        for parity in (1, 0):
            s_hashed = 3 if parity else 4
            s_inline = max(56 - e, 3)
            if s_inline % 2 != parity:
                s_inline += 1
            out.append((f"ext_{e}_{'odd' if parity else 'even'}_hashed",
                        lambda p, s=s_hashed, e=e: _ext(p, s, e, [_val(40, 1), _val(40, 2)], s & 1)))
            out.append((f"ext_{e}_{'odd' if parity else 'even'}_inline",
                        lambda p, s=s_inline, e=e: _ext(p, s, e, [b"\x01", b"\x02"], s & 1)))
    for t in sorted(EXT_TOTALS):
        out.append((f"ext_total_{t}", functools.partial(_tuned_ext, form=form, total=t)))
    return out


def _tuned_ext(pfx, form, total):
    # an extension of 8 nibbles (6 bytes of hex prefix) over an inline branch of 24 or 25 bytes
    for s in range(55, 2, -1):
        for other in (b"\x01", b"\x90"):
            items = _tune(lambda n: _ext(pfx, s, 8, [_val(n, 9), other], s & 1), form, "ext", s, total, range(1, 30))
            if items:
                return items
    raise AssertionError(f"no extension of {total} bytes")


def _shallow_gadgets():
    # fixed keys outside the two-nibble prefixes of the others (first nibbles 0, 1 and 15)
    return [
        ("leaf_63_nibbles", [(_key([0], 4), _val(5, 1)), (_key([15], 5), _val(6, 2))]),
        ("leaf_62_nibbles", [(_key([1, 0], 6), _val(7, 3)), (_key([1, 5], 7), b"\x7f")]),
    ]


@functools.lru_cache(maxsize=None)
def gadgets(form):
    """[(name, [(64 nibbles, value)])]: every gadget in `form`, each under its own prefix"""
    out = list(_shallow_gadgets())
    makers = _leaf_gadgets(form) + _branch_gadgets(form) + _ext_gadgets(form)
    makers.append(("root_single_leaf", lambda p: [(_key(p, 8), _val(3, 4))]))
    assert len(makers) <= 13 * 16
    for g, (name, make) in enumerate(makers):
        pfx = [2 + g // 16, g % 16]
        items = make(pfx)
        assert all(k[:2] == pfx and len(k) == 64 for k, _ in items), name
        out.append((name, sorted(items)))
    return out


def union(form):
    items = [it for _, its in gadgets(form) for it in its]
    assert len({tuple(k) for k, _ in items}) == len(items)
    return sorted(items)


def _bytes_key(nib):
    return bytes((nib[i] << 4) | nib[i + 1] for i in range(0, 64, 2))


def _arrays(items):
    keys = np.array([list(_bytes_key(k)) for k, _ in items], dtype=np.uint8).reshape(-1, 32)
    off = np.zeros(len(items) + 1, dtype=np.uint64)
    np.cumsum([len(v) for _, v in items], out=off[1:])
    vals = np.frombuffer(b"".join(v for _, v in items) or b"\0", dtype=np.uint8)[: int(off[-1])].copy()
    return keys, off, vals


def _model_root(items):
    return tm.keccak(tm.node_rlp(items, 0))


# ---------------------------------------------------------------- coverage ------------------------------------------
def _realized(form):
    got = set()
    for name, items_w in gadgets(form):
        model = _model_items(items_w, form)
        nodes = list(tm.walk(model))
        top = nodes[0]
        got.add(("root", top.kind))
        if top.kind == "ext" and top.nibble_count == 63:
            got.add(("root", "ext_over_last_nibble_branch"))
        for nd in nodes:
            pl = tm.payload_len(nd.encoded_len)
            if nd.kind == "leaf":
                got |= {("leaf_nibbles", nd.nibble_count), ("leaf_total", nd.encoded_len), ("payload", pl)}
            elif nd.kind == "branch":
                got |= {("branch_children", nd.n_children), ("branch_total", nd.encoded_len), ("branch_payload", pl),
                        ("slot0", 0 in nd.child_slots), ("slot15", 15 in nd.child_slots)}
                if 0 < len(nd.inline_child_slots) < nd.n_children:  # inline and hashed children mixed
                    got |= {("inline_at", j) for j, s in enumerate(nd.child_slots) if s in nd.inline_child_slots}
            else:
                got |= {("ext", nd.nibble_count, nd.start_nibble & 1, bool(nd.inline_child_slots)), ("ext_total", nd.encoded_len)}
        for _, w in items_w:  # the value as the encoder under test takes it
            got.add(("value_len", len(w)))
            if len(w) == 1:
                got.add(("one_byte", w[0]))
    return got


def _wanted():
    want = {("root", "leaf"), ("root", "ext"), ("root", "branch"), ("root", "ext_over_last_nibble_branch")}
    want |= {("leaf_nibbles", r) for r in LEAF_NIBBLES} | {("leaf_total", t) for t in LEAF_TOTALS}
    want |= {("payload", p) for p in LIST_PAYLOADS}
    want |= {("value_len", n) for n in VALUE_LENGTHS} | {("one_byte", b) for b in ONE_BYTE_VALUES}
    want |= {("branch_children", k) for k in range(2, 17)} | {("branch_total", t) for t in BRANCH_TOTALS}
    want |= {("branch_payload", p) for p in BRANCH_PAYLOADS}
    want |= {(s, present) for s in ("slot0", "slot15") for present in (True, False)}
    want |= {("inline_at", j) for j in range(16)}
    want |= {("ext", e, par, inl) for e in EXT_NIBBLES for par in (0, 1) for inl in (False, True)}
    want |= {("ext_total", t) for t in EXT_TOTALS}
    return want


@pytest.mark.parametrize("form", sorted(FORMS))
def test_gadgets_reach_every_encoding_boundary(form):
    missing = _wanted() - _realized(form)
    assert not missing, f"{form} gadgets miss: {sorted(missing, key=str)}"


def test_model_subtrie_top_lengths_by_depth():
    # one leaf with a one-byte value: its encoding shrinks by one byte every second nibble of depth
    item = [(_key([], 0), b"\x01")]
    assert [len(tm.node_rlp(item, d)) for d in range(1, 11)] == [35, 35, 34, 34, 33, 33, 32, 32, 31, 31]
    assert tm.subtrie_ref(item, 8) is not None and tm.subtrie_ref(item, 9) is None


# ---------------------------------------------------------------- oracle == model -----------------------------------
def test_oracle_equals_model_on_every_gadget_and_the_union(oracle):
    for name, items in gadgets("raw"):
        assert oracle.trie_root_from_leaves(*_arrays(items)) == _model_root(items), name
    items = union("raw")
    assert oracle.trie_root_from_leaves(*_arrays(items)) == _model_root(items)


# ---------------------------------------------------------------- witness form --------------------------------------
def _emit(items, depth, leaf_op):
    """the compact-witness instructions of the canonical trie over items [(nibbles, x)], children before parents"""
    if len(items) == 1:
        return leaf_op(items[0][0][depth:], items[0][1])
    cp = tm.common_depth(items, depth)
    if cp > depth:
        return _emit(items, cp, leaf_op) + ws.ext(items[0][0][depth:cp])
    out, mask = b"", 0
    for n, sub in enumerate(tm.split_children(items, depth)):
        if sub:
            out += _emit(sub, depth + 1, leaf_op)
            mask |= 1 << n
    return out + ws.branch(mask)


def _account_op(key_nibbles, nonce=0, balance=0, storage=None):
    """an account leaf: nonce / balance omitted when zero; storage: the stream of its storage trie (emitted first)"""
    flags = (2 if storage is not None else 0) | (4 if nonce else 0) | (8 if balance else 0)
    body = (synth.cbor_uint(nonce) if nonce else b"") + (synth.cbor_bytes(balance.to_bytes((balance.bit_length() + 7) // 8, "big")) if balance else b"")
    return (storage or b"") + bytes([ws.OP_ACCOUNT]) + synth.cbor_bytes(synth.compact_key(key_nibbles)) + bytes([flags]) + body


def _account_rlp(nonce, balance, storage_root):
    return synth.rlp_list([synth.rlp_int(nonce), synth.rlp_int(balance), synth.rlp_str(storage_root), synth.rlp_str(EMPTY_CODE_HASH)])


# nonce / balance at the edges of the significant-byte count and of the single-byte string rule
EDGE_INTS = [0, 1, 0x7F, 0x80, 0xFF, 0x100, (1 << 32) - 1, 1 << 32]


def _edge_accounts():
    """[(nonce, balance, r)]: account leaves with r key nibbles left; the last three are tuned to 135, 136, 137 bytes"""
    pairs = [(x, y) for x in EDGE_INTS for y in (x, EDGE_INTS[-1])]
    pairs += [((1 << 64) - 1, 5), (3, 1 << 255), (0, (1 << 256) - 1), ((1 << 64) - 1, (1 << 256) - 1)]
    accts = [(n, b, 1 + i % 5) for i, (n, b) in enumerate(pairs)]
    for total in (135, 136, 137):
        found = None
        for r in range(0, 61):
            for nonce in (0, 1, 0x80, 0x100, (1 << 32) - 1, 1 << 32, (1 << 64) - 1):
                for balance in ((1 << 256) - 1, 1 << 255, (1 << 248) - 1):
                    nib = _key([], r)
                    if len(tm.node_rlp([(nib, _account_rlp(nonce, balance, tm.EMPTY_TRIE_HASH))], 64 - r)) == total:
                        found = found or (nonce, balance, r)
        assert found, total
        accts.append(found)
    return accts


@functools.lru_cache(maxsize=None)
def witness_case():
    """(witness, model state root, {hashed address: model storage root}, [encoded lengths of the edge account leaves])"""
    state = []  # (64 nibbles, (op bytes without key, account rlp))
    storage_roots = {}
    for g, (name, items_w) in enumerate(gadgets("witness")):
        key = tm.nibbles(synth.keccak256(b"storage gadget %d" % g))
        model = _model_items(items_w, "witness")
        root = _model_root(model)
        stream = _emit(sorted(items_w), 0, lambda nib, w: ws.leaf(nib, w))
        state.append((key, (stream, 0, 7 + g, root)))
        storage_roots[_bytes_key(key)] = root
    hashed_storage = synth.keccak256(b"a storage trie given as a hash node")
    key = tm.nibbles(synth.keccak256(b"hash node storage"))
    state.append((key, (ws.hashnode(hashed_storage), 1, 1, hashed_storage)))
    storage_roots[_bytes_key(key)] = hashed_storage
    edge_keys = []
    for i, (nonce, balance, r) in enumerate(_edge_accounts()):
        # a pair below a branch at depth 63 - r, under its own first three nibbles (the gadget keys above are hashes)
        base = _fill([14, i // 16, i % 16], 63 - r, i)
        a, b = base + [3] + _key([], i)[:r], base + [12] + _key([], i + 1)[:r]
        state += [(a, (None, nonce, balance, tm.EMPTY_TRIE_HASH)), (b, (None, 1, 2, tm.EMPTY_TRIE_HASH))]
        edge_keys.append((a, 64 - r))
    state.sort()
    assert len({tuple(k) for k, _ in state}) == len(state)
    model = [(k, _account_rlp(n, b, root)) for k, (_, n, b, root) in state]
    wit = ws.HDR + _emit(state, 0, lambda nib, acc: _account_op(nib, acc[1], acc[2], acc[0]))
    lens = [len(tm.node_rlp([it for it in model if it[0] == k], d)) for k, d in edge_keys]
    return wit, _model_root(model), storage_roots, lens


def test_witness_form_gadgets_decode_in_the_oracle_to_the_model_roots(oracle):
    from ppd_oracle_lib import parse_pre_image_dump

    wit, state_root, storage_roots, lens = witness_case()
    assert {135, 136, 137} <= set(lens)
    d = parse_pre_image_dump(oracle.compact_decode(wit))
    assert d["state_root"] == state_root
    for k, root in storage_roots.items():
        assert d["storage"][k] == root


# ---------------------------------------------------------------- GPU: the sorted-leaves builder --------------------
@pytest.fixture(scope="module")
def ctx():
    from proof_protocol_decoder_b200.lib import Context

    c = Context(0)
    yield c
    c.close()


@pytest.mark.gpu
def test_sorted_leaves_builder_on_every_gadget(ctx, oracle):
    for name, items in gadgets("raw"):
        arrays = _arrays(items)
        want = _model_root(items)
        assert oracle.trie_root_from_leaves(*arrays) == want, name
        assert ctx.trie_root_sorted_leaves(*arrays) == want, name


@pytest.mark.gpu
@pytest.mark.parametrize("shift", [0, 1, 2, 3])
def test_sorted_leaves_builder_on_all_gadgets_at_once(ctx, oracle, shift):
    # lanes of every length, parity and value alignment in the same warps
    items = union("raw")
    keys, off, vals = _arrays(items)
    want = _model_root(items)
    if shift == 0:
        assert oracle.trie_root_from_leaves(keys, off, vals) == want
    shifted = np.concatenate([np.full(shift, 0xEE, np.uint8), vals])
    assert ctx.trie_root_sorted_leaves(keys, off + np.uint64(shift), shifted) == want


# ---------------------------------------------------------------- GPU: sub-tries and the top branch -----------------
def _subroot(ctx, items, base_depth):
    import torch

    keys, off, vals = _arrays(items)
    k = torch.from_numpy(keys).cuda()
    o = torch.from_numpy(off.astype(np.int64)).cuda()
    v = torch.from_numpy(vals if len(vals) else np.zeros(1, np.uint8)).cuda()
    return ctx.trie_subroot_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), len(items), int(off[-1]), base_depth)


def _part(base_depth, top):
    """a part below `base_depth` nibbles whose top node is a leaf, a branch or an extension of three nibbles"""
    base = _key([], 11)[:base_depth]
    if top == "leaf":
        return [(base + _key([], 1)[: 64 - base_depth], _val(40, 1))]
    if top == "branch":
        return sorted((base + [s] + _key([], s)[: 63 - base_depth], _val(3, s)) for s in (0, 7, 15))
    return sorted((base + [5, 6, 7, s] + _key([], s)[: 60 - base_depth], _val(3, s)) for s in (2, 9))


@pytest.mark.gpu
@pytest.mark.parametrize("top", ["leaf", "branch", "ext"])
@pytest.mark.parametrize("base_depth", [1, 2, 3, 8, 17, 40])
def test_subtrie_ref_equals_model(ctx, base_depth, top):
    items = _part(base_depth, top)
    assert next(tm.walk(items, base_depth)).kind == top
    want = tm.subtrie_ref(items, base_depth)
    assert want is not None
    assert _subroot(ctx, items, base_depth) == want


@pytest.mark.gpu
def test_subtrie_top_shorter_than_32_bytes_is_rejected(ctx):
    from proof_protocol_decoder_b200 import PpdError

    one = [(_key([], 0), b"\x01")]
    assert _subroot(ctx, one, 8) == tm.subtrie_ref(one, 8)  # exactly 32 bytes: hashed
    k63 = _key([], 0)[:63]
    short = [
        (one, 9),                                                  # a leaf of 31 bytes
        ([(k63[:62] + [1, 3], b"\x01"), (k63[:62] + [8, 4], b"\x01")], 62),  # a branch of 22 bytes
        ([(k63 + [2], b"\x01"), (k63 + [9], b"\x01")], 50),        # an extension of 31 bytes over an inline branch
    ]
    for items, depth in short:
        assert tm.subtrie_ref(items, depth) is None
        with pytest.raises(PpdError) as e:
            _subroot(ctx, items, depth)
        assert e.value.code == 62, (items, depth)


@pytest.mark.gpu
def test_subtrie_keys_not_sharing_the_base_nibbles_are_rejected(ctx):
    from proof_protocol_decoder_b200 import PpdError

    cases = [
        ([_key([0, 5], 1), _key([1, 5], 2)], 2),                      # no nibble in common
        ([_key([3, 0], 1), _key([3, 1], 2)], 2),                      # base_depth - 1 nibbles in common
        ([_key([7] * 8, 1), _key([7] * 8 + [9], 2), _key([7] * 4 + [8], 3)], 8),  # only the last pair breaks it
    ]
    for keys, depth in cases:
        items = sorted((k, b"\x01\x02") for k in keys)
        with pytest.raises(PpdError) as e:
            _subroot(ctx, items, depth)
        assert e.value.code == 62, depth


@pytest.mark.gpu
def test_top_branch_over_gathered_refs(ctx):
    from proof_protocol_decoder_b200 import PpdError

    refs = [synth.keccak256(b"part %d" % i) for i in range(16)]
    blob = b"".join(refs)
    for mask in (0x0003, 0x8001, 0xC000, 0x7FFE, 0xFFFF):
        kids = [synth.rlp_str(refs[i]) if (mask >> i) & 1 else b"\x80" for i in range(16)]
        assert ctx.trie_root_from_children(blob, mask) == synth.keccak256(synth.rlp_list(kids + [b"\x80"])), hex(mask)
    assert ctx.trie_root_from_children(blob, 0x10003) == ctx.trie_root_from_children(blob, 0x0003)
    for mask in (0, 0x0001, 0x8000, 0x10000, 0x10004):
        with pytest.raises(PpdError) as e:
            ctx.trie_root_from_children(blob, mask)
        assert e.value.code == 62, hex(mask)


@pytest.mark.gpu
@pytest.mark.parametrize("tops", [(3, 12), (0, 7, 15), tuple(n for n in range(16) if n != 6)], ids=["2", "3", "15"])
def test_split_with_partial_top_nibbles_equals_whole_trie(ctx, tops):
    import torch

    from proof_protocol_decoder_b200 import shard

    rng = np.random.default_rng(len(tops))
    raw = rng.integers(0, 256, (240, 32), dtype=np.uint8)
    raw[:, 0] = (np.array(tops, dtype=np.uint8)[rng.integers(0, len(tops), len(raw))] << 4) | (raw[:, 0] & 15)
    keys = sorted({r.tobytes() for r in raw})
    items = [(tm.nibbles(k), _val(int(rng.integers(1, 80)), i)) for i, k in enumerate(keys)]
    k_np, off, vals = _arrays(items)
    k = torch.from_numpy(k_np).cuda()
    o = torch.from_numpy(off.astype(np.int64)).cuda()
    v = torch.from_numpy(vals).cuda()
    whole = ctx.trie_root_sorted_leaves_dev(k.data_ptr(), o.data_ptr(), v.data_ptr(), len(items), int(off[-1]))
    refs, mask, _ = shard.split_trie_refs(ctx, torch, k, o, v)
    assert mask == sum(1 << t for t in tops)
    assert ctx.trie_root_from_children(b"".join(refs), mask) == whole == _model_root(items)


# ---------------------------------------------------------------- GPU: the arena level hasher -----------------------
def _with_env(name, on, fn):
    saved = os.environ.pop(name, None)
    if on:
        os.environ[name] = "1"
    try:
        return fn()
    finally:
        os.environ.pop(name, None)
        if saved is not None:
            os.environ[name] = saved


@pytest.mark.gpu
def test_arena_hasher_on_witness_gadgets_and_edge_accounts(ctx, oracle):
    from proof_protocol_decoder_b200 import flat

    wit, state_root, storage_roots, _ = witness_case()
    want = oracle.compact_decode(wit)
    for host_parse in (False, True):
        got, st = _with_env("PPD_HOST_PARSE", host_parse, lambda: (ctx.compact_decode(wit), ctx.stats()))
        assert st["witnesses_on_gpu"] == (0 if host_parse else 1)
        assert got == want, "host parser" if host_parse else "GPU parser"
        d = flat.parse_pre_image_dump(got)
        assert d["state_root"] == state_root
        assert {k: d["storage"][k] for k in storage_roots} == storage_roots


def _edge_value_block(seed):
    """a synth block whose traces write values at the RLP edges: balances 0, 0x7f, 0x80, 2^256 - 1, storage values
    0x01 .. 2^256 - 1, and one account's nonce going from 127 to 128"""
    blk = synth.gen_block(600 + seed, n_accounts=60, n_txns=4, contract_frac=0.6, slots_hi=16, slot_writes=(1, 6), allow_self_destruct=False)
    balances = [0, 0x7F, 0x80, (1 << 256) - 1]
    writes = [0x01, 0x7F, 0x80, 0xFF, 0x100, (1 << 256) - 1]
    nb = nw = 0
    for tx in blk.txns:
        for _, tr in tx["traces"]:
            if "balance" in tr:
                tr["balance"] = balances[nb % len(balances)]
                nb += 1
            if tr.get("storage_written"):
                tr["storage_written"] = [(k, writes[(nw + j) % len(writes)]) for j, (k, _) in enumerate(tr["storage_written"])]
                nw += len(tr["storage_written"])
    assert nb >= len(balances) and nw >= len(writes)
    addr, tr0 = blk.txns[0]["traces"][0]
    tr0["nonce"] = 127
    later = dict(blk.txns[1]["traces"])
    if addr in later:
        later[addr]["nonce"] = 128
    else:
        blk.txns[1]["traces"].append((addr, {"nonce": 128}))
    return blk


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_values_written_by_transactions_at_encoding_edges(ctx, oracle, seed):
    f = _edge_value_block(seed).flat
    want = oracle.block_decode(f)
    for host_txn in (False, True):
        got, st = _with_env("PPD_HOST_TXN", host_txn, lambda: (ctx.block_decode(f), ctx.stats()))
        assert got == want, "host txn loop" if host_txn else "device txn loop"
        if not host_txn:
            assert st["txn_loops_on_gpu"] == 1
