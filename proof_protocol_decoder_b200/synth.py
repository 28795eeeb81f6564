"""Synthetic inputs of the shapes BASELINE.json names (SURVEY.md 8d): compact witnesses plus
per-txn traces that are consistent with them, and sorted leaf sets for the rehash sweep.

Generators are pure numpy/Python and carry their own batch Keccak-256 (`keccak256_many`), so they
depend on neither the CUDA library nor the oracle; the same bytes are fed to both.
"""
import struct

import numpy as np

from . import flat

# ------------------------------------------------------------------------------------------------
# numpy Keccak-256 (rate 136, padding 0x01..0x80), vectorised over a batch of messages
# ------------------------------------------------------------------------------------------------
_RC = np.array(
    [
        0x0000000000000001, 0x0000000000008082, 0x800000000000808A, 0x8000000080008000, 0x000000000000808B, 0x0000000080000001,
        0x8000000080008081, 0x8000000000008009, 0x000000000000008A, 0x0000000000000088, 0x0000000080008009, 0x000000008000000A,
        0x000000008000808B, 0x800000000000008B, 0x8000000000008089, 0x8000000000008003, 0x8000000000008002, 0x8000000000000080,
        0x000000000000800A, 0x800000008000000A, 0x8000000080008081, 0x8000000000008080, 0x0000000080000001, 0x8000000080008008,
    ],
    dtype=np.uint64,
)
_ROT = [[0, 36, 3, 41, 18], [1, 44, 10, 45, 2], [62, 6, 43, 15, 61], [28, 55, 25, 21, 56], [27, 20, 39, 8, 14]]  # [x][y]


def _rotl(a, k):
    if k == 0:
        return a
    return (a << np.uint64(k)) | (a >> np.uint64(64 - k))


def _keccak_f(A):
    """A: uint64 [25, N], lane index x + 5 y."""
    for rnd in range(24):
        C = [A[x] ^ A[x + 5] ^ A[x + 10] ^ A[x + 15] ^ A[x + 20] for x in range(5)]
        D = [C[(x + 4) % 5] ^ _rotl(C[(x + 1) % 5], 1) for x in range(5)]
        B = [None] * 25
        for x in range(5):
            for y in range(5):
                B[y + 5 * ((2 * x + 3 * y) % 5)] = _rotl(A[x + 5 * y] ^ D[x], _ROT[x][y])
        for y in range(5):
            for x in range(5):
                A[x + 5 * y] = B[x + 5 * y] ^ (~B[(x + 1) % 5 + 5 * y] & B[(x + 2) % 5 + 5 * y])
        A[0] = A[0] ^ _RC[rnd]
    return A


def keccak256_many(msgs):
    """list of bytes -> np.uint8 [n, 32]"""
    n = len(msgs)
    out = np.zeros((n, 32), dtype=np.uint8)
    if n == 0:
        return out
    nblocks = np.array([len(m) // 136 + 1 for m in msgs])
    for nb in np.unique(nblocks):
        idx = np.nonzero(nblocks == nb)[0]
        buf = np.zeros((len(idx), nb * 136), dtype=np.uint8)
        for r, i in enumerate(idx):
            m = msgs[i]
            buf[r, : len(m)] = np.frombuffer(m, dtype=np.uint8)
            buf[r, len(m)] ^= 0x01
        buf[:, nb * 136 - 1] ^= 0x80
        lanes = buf.view("<u8").reshape(len(idx), nb, 17)
        A = [np.zeros(len(idx), dtype=np.uint64) for _ in range(25)]
        for b in range(nb):
            for k in range(17):
                A[k] = A[k] ^ lanes[:, b, k]
            A = _keccak_f(A)
        dig = np.stack(A[:4], axis=1).astype("<u8").view(np.uint8).reshape(len(idx), 32)
        out[idx] = dig
    return out


def keccak256_fixed(data):
    """np.uint8 [n, L] with L < 136 -> np.uint8 [n, 32]"""
    data = np.ascontiguousarray(data, dtype=np.uint8)
    n, L = data.shape
    assert L < 136
    buf = np.zeros((n, 136), dtype=np.uint8)
    buf[:, :L] = data
    buf[:, L] ^= 0x01
    buf[:, 135] ^= 0x80
    lanes = buf.view("<u8")
    A = [lanes[:, k].copy() if k < 17 else np.zeros(n, dtype=np.uint64) for k in range(25)]
    A = _keccak_f(A)
    return np.stack(A[:4], axis=1).astype("<u8").view(np.uint8).reshape(n, 32)


def keccak256(m: bytes) -> bytes:
    return keccak256_many([m])[0].tobytes()


# ------------------------------------------------------------------------------------------------
# encoders
# ------------------------------------------------------------------------------------------------
def cbor_head(major, v):
    if v < 24:
        return bytes([(major << 5) | v])
    if v < 256:
        return bytes([(major << 5) | 24, v])
    if v < 65536:
        return bytes([(major << 5) | 25]) + v.to_bytes(2, "big")
    if v < 1 << 32:
        return bytes([(major << 5) | 26]) + v.to_bytes(4, "big")
    return bytes([(major << 5) | 27]) + v.to_bytes(8, "big")


def cbor_bytes(b):
    return cbor_head(2, len(b)) + bytes(b)


def cbor_uint(v):
    return cbor_head(0, v)


def compact_key(nibbles):
    """Erigon compact key that compact_prestate_processing.rs:1338-1390 decodes back to `nibbles`."""
    k = len(nibbles)
    if k == 0:
        return b""
    odd = k & 1
    body = bytearray()
    for i in range(0, k - 1, 2):
        body.append((nibbles[i] << 4) | nibbles[i + 1])
    if odd:
        body.append(nibbles[-1] << 4)
    return bytes([0x02 | odd]) + bytes(body)


def rlp_str(b):
    b = bytes(b)
    if len(b) == 1 and b[0] < 0x80:
        return b
    if len(b) < 56:
        return bytes([0x80 + len(b)]) + b
    ll = (len(b).bit_length() + 7) // 8
    return bytes([0xB7 + ll]) + len(b).to_bytes(ll, "big") + b


def rlp_list(items):
    pl = b"".join(items)
    if len(pl) < 56:
        return bytes([0xC0 + len(pl)]) + pl
    ll = (len(pl).bit_length() + 7) // 8
    return bytes([0xF7 + ll]) + len(pl).to_bytes(ll, "big") + pl


def rlp_int(v):
    return rlp_str(v.to_bytes((v.bit_length() + 7) // 8, "big")) if v else b"\x80"


def legacy_receipt(status, cum_gas, n_logs, rng):
    logs = []
    for _ in range(n_logs):
        topics = rlp_list([rlp_str(rng.bytes(32)) for _ in range(int(rng.integers(0, 4)))])
        logs.append(rlp_list([rlp_str(rng.bytes(20)), topics, rlp_str(rng.bytes(int(rng.integers(0, 96))))]))
    return rlp_list([rlp_int(status), rlp_int(cum_gas), rlp_str(rng.bytes(256)), rlp_list(logs)])


# ------------------------------------------------------------------------------------------------
# witness emission
# ------------------------------------------------------------------------------------------------
_HEX = "0123456789abcdef"


class _Emitter:
    def __init__(self, rng, virtual_depth=0, virtual_fill=None):
        self.rng = rng
        self.out = []
        self.vdepth = virtual_depth
        self.vfill = virtual_fill or []
        self._pool = b""
        self._pp = 0

    def rand_hash(self):
        if self._pp + 32 > len(self._pool):
            self._pool = self.rng.bytes(32 * 65536)
            self._pp = 0
        h = self._pool[self._pp : self._pp + 32]
        self._pp += 32
        return h

    def emit(self, keys, lo, hi, depth, leaf_fn):
        """keys: sorted list of hex strings; leaf_fn(i, depth) appends the leaf's opcodes"""
        out = self.out
        if hi - lo == 1 and depth >= self.vdepth:
            leaf_fn(lo, depth)
            return
        if depth >= self.vdepth:
            a, b = keys[lo], keys[hi - 1]
            cp = depth
            while a[cp] == b[cp]:
                cp += 1
            if cp > depth:
                self.emit(keys, lo, hi, cp, leaf_fn)
                out.append(b"\x01" + cbor_bytes(compact_key([int(c, 16) for c in a[depth:cp]])))
                return
        mask = 0
        i = lo
        fill = self.vfill[depth] if depth < self.vdepth else 0.0
        for nib in range(16):
            ch = _HEX[nib]
            j = i
            while j < hi and keys[j][depth] == ch:
                j += 1
            if j > i:
                self.emit(keys, i, j, depth + 1, leaf_fn)
                mask |= 1 << nib
            elif fill and self.rng.random() < fill:
                out.append(b"\x03" + self.rand_hash())
                mask |= 1 << nib
            i = j
        out.append(b"\x02" + cbor_uint(mask))


# ------------------------------------------------------------------------------------------------
# block generator (configs 1-4)
# ------------------------------------------------------------------------------------------------
def _rand_addr(rng, n):
    """n distinct 20-byte addresses whose Keccak has a non-zero first byte (SURVEY.md 8c hazard 4)."""
    addrs, hashed = [], []
    while len(addrs) < n:
        cand = np.frombuffer(rng.bytes(20 * (n - len(addrs) + 8)), dtype=np.uint8).reshape(-1, 20)
        h = keccak256_fixed(cand)
        for a, hh in zip(cand, h):
            if hh[0] != 0 and len(addrs) < n:
                addrs.append(a.tobytes())
                hashed.append(hh.tobytes())
    return addrs, hashed


def _rand_slot_keys(rng, n):
    """raw slot keys with a non-zero first byte (both readings of Nibbles::bytes_be agree) + their hashes"""
    raw = np.frombuffer(rng.bytes(32 * n), dtype=np.uint8).reshape(n, 32).copy()
    raw[:, 0] |= 0x10
    return [r.tobytes() for r in raw], [h.tobytes() for h in keccak256_fixed(raw)]


class _SlotPool:
    """pre-hashed slot keys, generated in large batches"""

    def __init__(self, rng, chunk=4096):
        self.rng, self.chunk = rng, chunk
        self.raw, self.hashed = [], []

    def take(self, n):
        while len(self.raw) < n:
            r, h = _rand_slot_keys(self.rng, max(self.chunk, n))
            self.raw.extend(r)
            self.hashed.extend(h)
        r, h = self.raw[:n], self.hashed[:n]
        del self.raw[:n], self.hashed[:n]
        return r, h


class SynthBlock:
    """A generated block: `flat` (FlatBlock bytes) plus the pieces it was made of."""

    def __init__(self):
        self.compact = b""
        self.txns = []
        self.resolved_code = []
        self.withdrawals = []
        self.checkpoint = bytes(32)
        self.b_meta = b""
        self.b_hashes = b""
        self.stats = {}
        self.final_accounts = []

    @property
    def flat(self):
        return flat.encode_flat_block(self.compact, self.txns, self.resolved_code, self.withdrawals, self.checkpoint, self.b_meta, self.b_hashes)

    def to_block_trace(self):
        from .trace_protocol import BlockLevelData, BlockTrace, ContractCodeUsage, OtherBlockData, ProcessingMeta, TxnInfo, TxnMeta, TxnTrace

        infos = []
        for tx in self.txns:
            traces = {}
            for addr, d in tx["traces"]:
                cu = None
                if d.get("code_read") is not None:
                    cu = ContractCodeUsage(read=d["code_read"])
                elif d.get("code_write") is not None:
                    cu = ContractCodeUsage(write=d["code_write"])
                sw = dict(d["storage_written"]) if d.get("storage_written") is not None else None
                traces[addr] = TxnTrace(d.get("balance"), d.get("nonce"), d.get("storage_read"), sw, cu, d.get("self_destructed") or None)
            infos.append(TxnInfo(traces, TxnMeta(tx["byte_code"], tx["new_txn_trie_node_byte"], tx["new_receipt_trie_node_byte"], tx["gas_used"])))
        bt = BlockTrace({"combined": {"compact": self.compact}}, infos)
        code = dict(self.resolved_code)
        meta = ProcessingMeta(lambda h: code.get(h))  # None: the witness carries that code
        other = OtherBlockData(BlockLevelData(self.b_meta, self.b_hashes, list(self.withdrawals)), self.checkpoint)
        return bt, meta, other


def gen_block(
    seed,
    n_accounts=1000,
    n_txns=10,
    contract_frac=0.10,
    slots_lo=1,
    slots_hi=64,
    virtual_depth=0,
    virtual_accounts_log16=7,
    accounts_per_txn=(3, 8),
    slot_reads=(0, 8),
    slot_writes=(0, 8),
    allow_new_accounts=True,
    allow_self_destruct=True,
    inline_code_frac=0.2,
    n_withdrawals=0,
    zero_write_frac=0.10,
):
    """One BlockTrace of the C1/C2 shape.  virtual_depth > 0 embeds the accounts in a virtual state of
    16**virtual_accounts_log16 accounts: every branch above that depth gets its untouched siblings as
    random Hash opcodes with the occupancy of a uniform trie (so paths look like mainnet proofs)."""
    rng = np.random.default_rng(seed)
    blk = SynthBlock()
    pool = _SlotPool(rng)
    addrs, haddrs = _rand_addr(rng, n_accounts)
    order = sorted(range(n_accounts), key=lambda i: haddrs[i])
    accounts = []
    for i in range(n_accounts):
        acc = {
            "addr": addrs[i],
            "haddr": haddrs[i],
            "nonce": int(rng.integers(0, 1 << 16)),
            "balance": int.from_bytes(rng.bytes(12), "big"),
            "contract": bool(rng.random() < contract_frac),
            "slots": {},
            "alive": True,
        }
        if acc["contract"]:
            n_slots = int(np.exp(rng.uniform(np.log(slots_lo), np.log(slots_hi + 1))))
            n_slots = max(slots_lo, min(slots_hi, n_slots))
            raw, hashed = pool.take(n_slots)
            for rk, hk in zip(raw, hashed):
                vlen = int(rng.integers(1, 33))
                v = int.from_bytes(rng.bytes(vlen), "big") | 1
                acc["slots"][rk] = (hk, v)
            if rng.random() < inline_code_frac:
                acc["code"] = rng.bytes(int(rng.integers(1, 600)))
                acc["code_hash"] = keccak256(acc["code"])
            else:
                acc["code"] = None
                acc["code_hash"] = rng.bytes(32)
        accounts.append(acc)

    # ---- witness ----
    vfill = [1.0 - float(np.exp(-(16.0**virtual_accounts_log16) / 16.0 ** (d + 1))) for d in range(virtual_depth)]
    em = _Emitter(rng, virtual_depth, vfill)
    keys = [haddrs[i].hex() + "0" for i in order]  # sentinel char keeps a[cp] in range

    def storage_leaf_fn_for(skeys, svals):
        def fn(i, depth):
            nib = [int(c, 16) for c in skeys[i][depth:64]]
            v = svals[i]
            em.out.append(b"\x00" + cbor_bytes(compact_key(nib)) + cbor_bytes(v.to_bytes((v.bit_length() + 7) // 8, "big")))

        return fn

    def account_leaf_fn(i, depth):
        acc = accounts[order[i]]
        flags = 0
        if acc["contract"]:
            flags |= 1
            if acc["code"] is not None:
                em.out.append(b"\x04" + cbor_bytes(acc["code"]))
            else:
                em.out.append(b"\x03" + acc["code_hash"])
            if acc["slots"]:
                flags |= 2
                items = sorted((hk.hex() + "0", v) for (hk, v) in acc["slots"].values())
                sk = [k for k, _ in items]
                sv = [v for _, v in items]
                saved = em.vdepth
                em.vdepth = 0
                em.emit(sk, 0, len(sk), 0, storage_leaf_fn_for(sk, sv))
                em.vdepth = saved
        body = b""
        if acc["nonce"]:
            flags |= 4
            body += cbor_uint(acc["nonce"])
        if acc["balance"]:
            flags |= 8
            b = acc["balance"]
            body += cbor_bytes(b.to_bytes((b.bit_length() + 7) // 8, "big"))
        if flags & 1:
            body += cbor_uint(len(acc["code"]) if acc["code"] is not None else 1234)
        nib = [int(c, 16) for c in keys[i][depth:64]]
        em.out.append(b"\x05" + cbor_bytes(compact_key(nib)) + bytes([flags]) + body)

    em.out.append(b"\x01")
    if n_accounts:
        em.emit(keys, 0, len(keys), 0, account_leaf_fn)
    blk.compact = b"".join(em.out)

    # ---- traces ----
    code_table = {}
    cum_gas = 0
    live = list(range(n_accounts))
    for t in range(n_txns):
        k = int(rng.integers(accounts_per_txn[0], accounts_per_txn[1] + 1))
        k = min(k, len(live))
        picked = [live[j] for j in rng.choice(len(live), size=k, replace=False)] if k else []
        traces = []
        for pos, ai in enumerate(picked):
            acc = accounts[ai]
            tr = {}
            if pos == 0:
                acc["nonce"] += 1
                tr["nonce"] = acc["nonce"]
            if pos == 0 or rng.random() < 0.6:
                acc["balance"] = int.from_bytes(rng.bytes(12), "big")
                tr["balance"] = acc["balance"]
            if acc["contract"]:
                existing = list(acc["slots"].keys())
                nr = int(rng.integers(slot_reads[0], slot_reads[1] + 1))
                reads = []
                for _ in range(nr):
                    if existing and rng.random() < 0.85:
                        reads.append(existing[int(rng.integers(0, len(existing)))])
                    else:
                        reads.append(pool.take(1)[0][0])  # a slot that does not exist
                if reads or rng.random() < 0.3:
                    tr["storage_read"] = reads
                nw = int(rng.integers(slot_writes[0], slot_writes[1] + 1))
                writes = {}
                for _ in range(nw):
                    r = rng.random()
                    if existing and r < zero_write_frac:
                        kx = existing[int(rng.integers(0, len(existing)))]
                        writes[kx] = 0
                    elif existing and r < 0.6:
                        kx = existing[int(rng.integers(0, len(existing)))]
                        writes[kx] = int.from_bytes(rng.bytes(int(rng.integers(1, 33))), "big") | 1
                    else:
                        raw, hashed = pool.take(1)
                        writes[raw[0]] = int.from_bytes(rng.bytes(int(rng.integers(1, 33))), "big") | 1
                        acc["slots"][raw[0]] = (hashed[0], writes[raw[0]])
                for kx, v in writes.items():
                    if v == 0:
                        acc["slots"].pop(kx, None)
                    elif kx in acc["slots"]:
                        acc["slots"][kx] = (acc["slots"][kx][0], v)
                if writes:
                    tr["storage_written"] = list(writes.items())
                if rng.random() < 0.5:
                    tr["code_read"] = acc["code_hash"]
                    if acc["code"] is None:
                        code_table.setdefault(acc["code_hash"], rng.bytes(int(rng.integers(1, 400))))
                    elif ai >= n_accounts:  # created in this block: its code is not carried by the witness
                        code_table.setdefault(acc["code_hash"], acc["code"])
                if allow_self_destruct and pos > 0 and rng.random() < 0.03:
                    tr["self_destructed"] = True
                    acc["alive"] = False
            traces.append((acc["addr"], tr))
        if allow_new_accounts and rng.random() < 0.7:
            na, nh = _rand_addr(rng, 1)
            acc = {"addr": na[0], "haddr": nh[0], "nonce": 0, "balance": int.from_bytes(rng.bytes(10), "big") | 1, "contract": False, "slots": {}, "alive": True}
            tr = {"balance": acc["balance"]}
            if rng.random() < 0.4:  # contract creation
                code = rng.bytes(int(rng.integers(1, 500)))
                acc["contract"] = True
                acc["code"] = code
                acc["code_hash"] = keccak256(code)
                tr["code_write"] = code
                tr["nonce"] = 1
                acc["nonce"] = 1
                raw, hashed = pool.take(int(rng.integers(1, 5)))
                w = []
                for rk, hk in zip(raw, hashed):
                    v = int.from_bytes(rng.bytes(int(rng.integers(1, 33))), "big") | 1
                    acc["slots"][rk] = (hk, v)
                    w.append((rk, v))
                tr["storage_written"] = w
            accounts.append(acc)
            live.append(len(accounts) - 1)
            traces.append((acc["addr"], tr))
        live = [i for i in live if accounts[i]["alive"]]
        # the reference iterates a HashMap here: any order is legal
        perm = rng.permutation(len(traces))
        traces = [traces[j] for j in perm]
        gas = int(rng.integers(21000, 500001))
        cum_gas += gas
        rec = legacy_receipt(1, cum_gas, int(rng.integers(0, 3)), rng)
        if rng.random() < 0.3:
            rec = rlp_str(b"\x02" + rec)
        blk.txns.append(
            {
                "traces": traces,
                "byte_code": rng.bytes(int(rng.integers(110, 301))),
                "new_txn_trie_node_byte": b"",
                "new_receipt_trie_node_byte": rec,
                "gas_used": gas,
            }
        )
    blk.resolved_code = sorted(code_table.items())
    for _ in range(n_withdrawals):
        if not live:
            break
        acc = accounts[live[int(rng.integers(0, len(live)))]]
        blk.withdrawals.append((acc["addr"], int(rng.integers(1, 1 << 40))))
    blk.checkpoint = rng.bytes(32)
    blk.b_meta = rng.bytes(64)
    blk.b_hashes = rng.bytes(96)
    blk.stats = {"accounts": n_accounts, "txns": n_txns, "witness_bytes": len(blk.compact)}
    blk.final_accounts = accounts  # every account as the txns leave it (tests: an independent model of the final state)
    return blk


# ------------------------------------------------------------------------------------------------
# config 3: a storage-heavy block (few contracts with very large storage tries)
# ------------------------------------------------------------------------------------------------
_NIB = {c: i for i, c in enumerate(_HEX)}


def emit_full_trie(keys, leaf_bytes):
    """Witness stream (post-order, as compact_prestate_processing.rs:387-668 consumes it) of the FULL trie over
    `keys` (uint8 [n, 32], strictly ascending); leaf_bytes(i, key_suffix_hex) returns the leaf's instruction bytes.
    Iterative (one pass over the leaves with a stack of open branches): a million leaves take seconds."""
    n = len(keys)
    out = []
    if n == 0:
        return [b"\x06"]
    hexs = [k.tobytes().hex() for k in keys]
    if n == 1:
        return [leaf_bytes(0, hexs[0])]
    diff = keys[1:] != keys[:-1]
    first = diff.argmax(axis=1)
    assert diff.any(axis=1).all(), "keys must be distinct"
    x = keys[1:][np.arange(n - 1), first] ^ keys[:-1][np.arange(n - 1), first]
    lcp = (2 * first + (x < 16)).astype(np.int64)
    L = [-1] + lcp.tolist() + [-1]
    stack = []  # open branches: [depth, mask]
    for i in range(n):
        lc, ln = L[i], L[i + 1]
        hx = hexs[i]
        s = (lc if lc > ln else ln) + 1
        out.append(leaf_bytes(i, hx[s:]))
        if ln > lc:
            stack.append([ln, 1 << _NIB[hx[ln]]])
            continue
        stack[-1][1] |= 1 << _NIB[hx[lc]]
        while stack and stack[-1][0] > ln:
            d, mask = stack.pop()
            out.append(b"\x02" + cbor_uint(mask))
            parent = stack[-1][0] if stack else -1
            p = parent if parent > ln else ln
            if p < d - 1:
                ext = hx[p + 1 : d]
                out.append(b"\x01" + cbor_bytes(bytes([0x02 | (len(ext) & 1)]) + bytes.fromhex(ext + ("0" if len(ext) & 1 else ""))))
            if p < 0:
                break
            if stack and p == parent:
                stack[-1][1] |= 1 << _NIB[hx[p]]
            else:
                stack.append([p, 1 << _NIB[hx[p]]])
                break
    return out


def gen_c3_block(seed=3, n_contracts=4, slots=1_000_000, n_plain=1000, writes_per_contract=10_000, reads_per_contract=100):
    """BASELINE.json configs[2] / SURVEY.md 8d C3: `n_contracts` contracts with `slots` storage slots each (full leaves,
    values 1..32 bytes) plus `n_plain` plain accounts; ONE txn that writes `writes_per_contract` slots of every contract
    (60 % overwrite an existing slot, 10 % delete one, 30 % create a new one) and reads a few.  Only the slots the txn
    overwrites / deletes / reads need a known pre-image; the other leaves' keys are random 32-byte strings."""
    rng = np.random.default_rng(seed)
    blk = SynthBlock()
    n_acc = n_contracts + n_plain
    addrs, haddrs = _rand_addr(rng, n_acc)
    order = sorted(range(n_acc), key=lambda i: haddrs[i])
    contracts = list(range(n_contracts))
    known = min(slots, writes_per_contract + reads_per_contract)
    storage_streams, known_raw = {}, {}
    for c in contracts:
        raw, hashed = _rand_slot_keys(rng, known)
        rest = np.frombuffer(rng.bytes(32 * (slots - known)), dtype=np.uint8).reshape(-1, 32)
        keys = np.concatenate([np.frombuffer(b"".join(hashed), dtype=np.uint8).reshape(-1, 32), rest]) if known else rest
        be = keys.view(">u8")
        idx = np.lexsort((be[:, 3], be[:, 2], be[:, 1], be[:, 0]))
        keys = np.ascontiguousarray(keys[idx])
        vlen = rng.integers(1, 33, size=slots)
        vraw = rng.bytes(32 * slots)

        def leaf_bytes(i, suffix, vlen=vlen, vraw=vraw):
            v = bytes([vraw[32 * i] | 1]) + vraw[32 * i + 1 : 32 * i + int(vlen[i])]  # no leading zero byte
            k = bytes([0x02 | (len(suffix) & 1)]) + bytes.fromhex(suffix + ("0" if len(suffix) & 1 else "")) if suffix else b""
            return b"\x00" + cbor_bytes(k) + cbor_bytes(v)

        storage_streams[c] = emit_full_trie(keys, leaf_bytes)
        known_raw[c] = raw
    accounts = [{"addr": addrs[i], "nonce": int(rng.integers(0, 1 << 16)), "balance": int.from_bytes(rng.bytes(12), "big") | 1, "code_hash": rng.bytes(32)} for i in range(n_acc)]
    em = _Emitter(rng)
    keys_hex = [haddrs[i].hex() + "0" for i in order]

    def account_leaf_fn(i, depth):
        ai = order[i]
        acc = accounts[ai]
        flags = 4 | 8
        if ai < n_contracts:
            flags |= 1 | 2
            em.out.append(b"\x03" + acc["code_hash"])
            em.out.extend(storage_streams[ai])
        body = cbor_uint(acc["nonce"] or 1) + cbor_bytes(acc["balance"].to_bytes((acc["balance"].bit_length() + 7) // 8, "big"))
        if flags & 1:
            body += cbor_uint(1234)
        nib = [int(ch, 16) for ch in keys_hex[i][depth:64]]
        em.out.append(b"\x05" + cbor_bytes(compact_key(nib)) + bytes([flags]) + body)

    em.out.append(b"\x01")
    em.emit(keys_hex, 0, n_acc, 0, account_leaf_fn)
    blk.compact = b"".join(em.out)
    # ---- the txn ----
    sender = n_contracts  # a plain account
    traces = [(addrs[sender], {"nonce": accounts[sender]["nonce"] + 1, "balance": 12345})]
    for c in contracts:
        raw = known_raw[c]
        n_over, n_del = int(0.6 * writes_per_contract), int(0.1 * writes_per_contract)
        n_over, n_del = min(n_over, len(raw)), min(n_del, max(0, len(raw) - int(0.6 * writes_per_contract)))
        n_new = writes_per_contract - n_over - n_del
        new_raw, _ = _rand_slot_keys(rng, n_new)
        written = [(k, int.from_bytes(rng.bytes(int(rng.integers(1, 33))), "big") | 1) for k in raw[:n_over]]
        written += [(k, 0) for k in raw[n_over : n_over + n_del]]
        written += [(k, int.from_bytes(rng.bytes(int(rng.integers(1, 33))), "big") | 1) for k in new_raw]
        reads = raw[n_over + n_del : n_over + n_del + reads_per_contract]
        traces.append((addrs[c], {"balance": 777 + c, "storage_read": list(reads), "storage_written": written}))
    rec = legacy_receipt(1, 4_000_000, 2, rng)
    blk.txns.append({"traces": traces, "byte_code": rng.bytes(200), "new_txn_trie_node_byte": b"", "new_receipt_trie_node_byte": rec, "gas_used": 4_000_000})
    blk.stats = {"contracts": n_contracts, "slots": slots, "plain": n_plain, "writes_per_contract": writes_per_contract}
    return blk


def gen_config(name, seed=None):
    """The named BASELINE.json configs (scaled variants via kwargs of gen_block)."""
    if name == "C1":
        return gen_block(1 if seed is None else seed, n_accounts=1000, n_txns=10, n_withdrawals=2)
    if name == "C2":
        return gen_block(
            2 if seed is None else seed,
            n_accounts=20000,
            n_txns=200,
            contract_frac=0.15,
            slots_lo=1,
            slots_hi=4096,
            virtual_depth=7,
            accounts_per_txn=(80, 120),
            slot_reads=(0, 3),
            slot_writes=(0, 3),
            allow_new_accounts=False,
            allow_self_destruct=False,
            inline_code_frac=0.02,
        )
    if name == "C3":
        return gen_c3_block(3 if seed is None else seed)
    raise ValueError(name)


# ------------------------------------------------------------------------------------------------
# sorted leaves (config 5; storage-heavy tries of config 3)
# ------------------------------------------------------------------------------------------------
def gen_sorted_leaves(n, seed=5, val_lo=70, val_hi=80):
    """n distinct 32-byte keys in ascending order with account-RLP-shaped values of val_lo..val_hi bytes.
    Returns (keys uint8 [n,32], val_off uint64 [n+1], vals uint8)."""
    rng = np.random.default_rng(seed)
    keys = np.frombuffer(rng.bytes(32 * n), dtype=np.uint8).reshape(n, 32)
    be = keys.view(">u8")
    idx = np.lexsort((be[:, 3], be[:, 2], be[:, 1], be[:, 0]))
    keys = np.ascontiguousarray(keys[idx])
    if n > 1:
        assert (keys[1:] != keys[:-1]).any(axis=1).all()
    lens = rng.integers(val_lo, val_hi + 1, size=n).astype(np.uint64)
    val_off = np.zeros(n + 1, dtype=np.uint64)
    np.cumsum(lens, out=val_off[1:])
    vals = np.frombuffer(rng.bytes(int(val_off[-1])), dtype=np.uint8).copy()
    # shape the values as rlp lists: f8 <len-2> ... (content is opaque to the trie)
    vals[val_off[:-1].astype(np.int64)] = 0xF8
    vals[val_off[:-1].astype(np.int64) + 1] = (lens - 2).astype(np.uint8)
    return keys, val_off, vals


def gen_sorted_leaves_dev(n, seed=5, val_lo=70, val_hi=80, device="cuda"):
    """gen_sorted_leaves on the device (torch), for sizes the host generator is too slow for: n distinct 32-byte keys,
    ascending by construction (word 0 = i * step + r with 0 <= r < step; bytes 8..31 random), values of val_lo..val_hi
    random bytes.  Returns (keys uint8 [n,32], val_off int64 [n+1], vals uint8) on `device`."""
    import torch

    g = torch.Generator(device=device)
    g.manual_seed(seed)
    step = (1 << 62) // max(n, 1)
    w0 = torch.arange(n, dtype=torch.int64, device=device) * step + torch.randint(0, step, (n,), generator=g, device=device, dtype=torch.int64)
    keys = torch.randint(0, 256, (n, 32), generator=g, device=device, dtype=torch.uint8)
    sh = torch.arange(56, -8, -8, device=device, dtype=torch.int64)
    keys[:, :8] = ((w0[:, None] >> sh) & 0xFF).to(torch.uint8)
    lens = torch.randint(val_lo, val_hi + 1, (n,), generator=g, device=device, dtype=torch.int64)
    val_off = torch.zeros(n + 1, dtype=torch.int64, device=device)
    torch.cumsum(lens, 0, out=val_off[1:])
    vals = torch.randint(0, 256, (int(val_off[-1]),), generator=g, device=device, dtype=torch.uint8)
    return keys, val_off, vals


def permute_leaves_dev(keys, val_off, vals, perm, chunk=1 << 23):
    """The leaves (keys, val_off, vals) in the order perm (leaf j of the result is leaf perm[j]), values repacked
    (chunk leaves at a time: the byte-index temporaries stay a few GB at 100 M leaves)."""
    import torch

    lens = (val_off[1:] - val_off[:-1])[perm]
    off = torch.zeros_like(val_off)
    torch.cumsum(lens, 0, out=off[1:])
    out = torch.empty(int(off[-1]), dtype=torch.uint8, device=vals.device)
    for a in range(0, len(perm), chunk):
        b = min(a + chunk, len(perm))
        lo, hi = int(off[a]), int(off[b])
        src = torch.repeat_interleave(val_off[:-1][perm[a:b]] - off[a:b], lens[a:b], output_size=hi - lo)
        src += torch.arange(lo, hi, device=vals.device, dtype=torch.int64)
        out[lo:hi] = vals[src]
    return keys[perm].contiguous(), off, out
