"""FlatBlock writer and IrDump / PreImageDump readers (layouts: include/ppd_flat.h)."""
import struct

FLAT_BLOCK_MAGIC = 0x42445050
IR_DUMP_MAGIC = 0x49445050
PRE_IMAGE_MAGIC = 0x50445050

TR_BALANCE, TR_NONCE, TR_STORAGE_READ, TR_STORAGE_WRITTEN = 0x01, 0x02, 0x04, 0x08
TR_CODE_READ, TR_CODE_WRITE, TR_SELF_DESTRUCTED = 0x10, 0x20, 0x40

NODE_EMPTY, NODE_HASH, NODE_BRANCH, NODE_EXTENSION, NODE_LEAF = 0, 1, 2, 3, 4


def u256(v: int) -> bytes:
    return int(v).to_bytes(32, "big")


def _bytes(b) -> bytes:
    b = bytes(b)
    return struct.pack("<I", len(b)) + b


PRE_IMAGE_COMBINED, PRE_IMAGE_DIRECT = 0, 2


def encode_node(node) -> bytes:
    """A trie in the pre-order Node form of include/ppd_flat.h, from the tuples `parse_ir_dump` gives:
    ("empty",) | ("hash", h32) | ("branch", [16 nodes], value) | ("extension", nibbles, node) | ("leaf", nibbles, value)."""
    k = node[0]
    if k == "empty":
        return bytes([NODE_EMPTY])
    if k == "hash":
        assert len(node[1]) == 32
        return bytes([NODE_HASH]) + bytes(node[1])
    if k == "branch":
        assert len(node[1]) == 16
        return bytes([NODE_BRANCH]) + b"".join(encode_node(c) for c in node[1]) + _bytes(node[2])
    if k == "extension":
        return bytes([NODE_EXTENSION, len(node[1])]) + bytes(node[1]) + encode_node(node[2])
    if k == "leaf":
        return bytes([NODE_LEAF, len(node[1])]) + bytes(node[1]) + _bytes(node[2])
    raise ValueError("bad node %r" % (k,))


def encode_direct_pre_image(state_trie, storage_tries) -> bytes:
    """DirectPreImage payload (pre_image_kind 2): the state trie, then a trie per hashed address, sorted by address.
    Tries are node tuples (see encode_node) or already encoded bytes."""
    enc = lambda t: bytes(t) if isinstance(t, (bytes, bytearray, memoryview)) else encode_node(t)  # noqa: E731
    items = sorted((bytes(h), t) for h, t in (storage_tries.items() if isinstance(storage_tries, dict) else storage_tries))
    out = [enc(state_trie), struct.pack("<I", len(items))]
    for h, t in items:
        assert len(h) == 32
        out.append(h + enc(t))
    return b"".join(out)


def parse_direct_pre_image(b: bytes):
    """-> (state trie, {hashed address: trie}) as node tuples"""
    r = _R(b)
    state = _node(r)
    storage = {}
    for _ in range(r.u32()):
        h = r.take(32)
        storage[h] = _node(r)
    assert r.p == len(b), "trailing bytes in DirectPreImage"
    return state, storage


def with_pre_image(flat_block: bytes, kind: int, payload: bytes) -> bytes:
    """`flat_block` with its pre-image replaced (kind: PRE_IMAGE_COMBINED with TrieCompact bytes, PRE_IMAGE_DIRECT with
    a DirectPreImage payload)."""
    magic, ver, _kind, n = struct.unpack_from("<IIII", flat_block, 0)
    assert magic == FLAT_BLOCK_MAGIC and ver == 1
    return struct.pack("<III", magic, ver, kind) + _bytes(payload) + bytes(flat_block[16 + n :])


def pre_image_of(flat_block: bytes):
    """-> (kind, payload) of a FlatBlock"""
    magic, ver, kind, n = struct.unpack_from("<IIII", flat_block, 0)
    assert magic == FLAT_BLOCK_MAGIC and ver == 1
    return kind, bytes(flat_block[16 : 16 + n])


def encode_flat_block(compact, txns, resolved_code, withdrawals, checkpoint_state_trie_root, b_meta=b"", b_hashes=b"", pre_image_kind=PRE_IMAGE_COMBINED) -> bytes:
    """txns: list of dicts {traces: [(addr20, trace dict)], byte_code, new_txn_trie_node_byte,
    new_receipt_trie_node_byte, gas_used}; trace dict keys: balance, nonce (int or None),
    storage_read (list of 32-byte keys or None), storage_written (list of (key32, int value) or None),
    code_read (32-byte hash) | code_write (bytes), self_destructed (bool).
    `compact`: the TrieCompact bytes, or with pre_image_kind=PRE_IMAGE_DIRECT a DirectPreImage payload."""
    out = [struct.pack("<III", FLAT_BLOCK_MAGIC, 1, pre_image_kind), _bytes(compact), struct.pack("<I", len(txns))]
    for tx in txns:
        out.append(struct.pack("<I", len(tx["traces"])))
        for addr, tr in tx["traces"]:
            flags = 0
            body = []
            if tr.get("balance") is not None:
                flags |= TR_BALANCE
                body.append(u256(tr["balance"]))
            if tr.get("nonce") is not None:
                flags |= TR_NONCE
                body.append(u256(tr["nonce"]))
            if tr.get("storage_read") is not None:
                flags |= TR_STORAGE_READ
                body.append(struct.pack("<I", len(tr["storage_read"])))
                body.extend(bytes(k) for k in tr["storage_read"])
            if tr.get("storage_written") is not None:
                flags |= TR_STORAGE_WRITTEN
                body.append(struct.pack("<I", len(tr["storage_written"])))
                for k, v in tr["storage_written"]:
                    body.append(bytes(k) + u256(v))
            if tr.get("code_read") is not None:
                flags |= TR_CODE_READ
                body.append(bytes(tr["code_read"]))
            elif tr.get("code_write") is not None:
                flags |= TR_CODE_WRITE
                body.append(_bytes(tr["code_write"]))
            if tr.get("self_destructed"):
                flags |= TR_SELF_DESTRUCTED
            assert len(addr) == 20
            out.append(bytes(addr) + bytes([flags]) + b"".join(body))
        out.append(_bytes(tx.get("byte_code", b"")))
        out.append(_bytes(tx.get("new_txn_trie_node_byte", b"")))
        out.append(_bytes(tx.get("new_receipt_trie_node_byte", b"")))
        out.append(struct.pack("<Q", tx.get("gas_used", 0)))
    out.append(struct.pack("<I", len(resolved_code)))
    for h, code in resolved_code:
        out.append(bytes(h) + _bytes(code))
    out.append(struct.pack("<I", len(withdrawals)))
    for addr, amt in withdrawals:
        out.append(bytes(addr) + u256(amt))
    out.append(bytes(checkpoint_state_trie_root))
    out.append(_bytes(b_meta))
    out.append(_bytes(b_hashes))
    return b"".join(out)


class _R:
    def __init__(self, b):
        self.b, self.p = b, 0

    def take(self, n):
        v = self.b[self.p : self.p + n]
        assert len(v) == n, "dump truncated"
        self.p += n
        return v

    def u8(self):
        return self.take(1)[0]

    def u32(self):
        return struct.unpack("<I", self.take(4))[0]

    def u64(self):
        return struct.unpack("<Q", self.take(8))[0]

    def bytes_(self):
        return self.take(self.u32())


def _node(r):
    k = r.u8()
    if k == NODE_EMPTY:
        return ("empty",)
    if k == NODE_HASH:
        return ("hash", r.take(32))
    if k == NODE_BRANCH:
        ch = [_node(r) for _ in range(16)]
        return ("branch", ch, r.bytes_())
    if k == NODE_EXTENSION:
        n = r.u8()
        nib = list(r.take(n))
        return ("extension", nib, _node(r))
    if k == NODE_LEAF:
        n = r.u8()
        nib = list(r.take(n))
        return ("leaf", nib, r.bytes_())
    raise ValueError("bad node kind %d" % k)


def parse_trie(b: bytes):
    """One Trie in the pre-order Node form (a DirectPreImage's state trie, what ppd_trie_subset_* return) -> node tuple
    (see encode_node)"""
    r = _R(b)
    t = _node(r)
    assert r.p == len(b), "trailing bytes after the Trie"
    return t


def parse_ir_dump(b: bytes):
    """-> list of dicts mirroring plonky2_evm GenerationInputs (decoding.rs:131-145)."""
    r = _R(b)
    assert r.u32() == IR_DUMP_MAGIC
    out = []
    for _ in range(r.u32()):
        g = {}
        g["txn_number_before"] = int.from_bytes(r.take(32), "big")
        g["gas_used_before"] = int.from_bytes(r.take(32), "big")
        g["gas_used_after"] = int.from_bytes(r.take(32), "big")
        has = r.u8()
        st = r.bytes_()
        g["signed_txn"] = st if has else None
        g["withdrawals"] = [(r.take(20), int.from_bytes(r.take(32), "big")) for _ in range(r.u32())]
        tries = {"state_trie": _node(r), "transactions_trie": _node(r), "receipts_trie": _node(r)}
        tries["storage_tries"] = [(r.take(32), _node(r)) for _ in range(r.u32())]
        g["tries"] = tries
        g["trie_roots_after"] = {"state_root": r.take(32), "transactions_root": r.take(32), "receipts_root": r.take(32)}
        g["checkpoint_state_trie_root"] = r.take(32)
        g["contract_code"] = {r.take(32): r.bytes_() for _ in range(r.u32())}
        g["block_metadata"] = r.bytes_()
        g["block_hashes"] = r.bytes_()
        out.append(g)
    assert r.p == len(b), "trailing bytes in IrDump"
    return out


def parse_pre_image_dump(b: bytes):
    r = _R(b)
    assert r.u32() == PRE_IMAGE_MAGIC
    d = {"version": r.u8(), "state_root": r.take(32)}
    d["storage"] = {r.take(32): r.take(32) for _ in range(r.u32())}
    d["code"] = {}
    for _ in range(r.u32()):
        h = r.take(32)
        d["code"][h] = r.u32()
    d["nodes_hashed"] = r.u64()
    d["perms"] = r.u64()
    return d
