"""The canonical Merkle-Patricia trie as a recursive pure-Python model: an independent reference for the CUDA trie hashers.

A trie's shape is a function of its key set, so the model builds each node straight from the sorted items below it:
no insert, no delete, no collapse rule, and no code shared with the CUDA kernels or the C++ oracle (hashing is the numpy
Keccak of `synth`).  Items are [(nibbles, value)] sorted by nibbles, every key 64 nibbles long."""
import functools
from collections import namedtuple

from proof_protocol_decoder_b200 import synth

EMPTY_TRIE_HASH = synth.keccak256(b"\x80")


@functools.lru_cache(maxsize=1 << 14)
def keccak(raw):
    """keccak256, cached"""
    # cached: the edge-case generators re-encode the same children while they search for a value length
    return synth.keccak256(raw)


def nibbles(key):
    return [x for b in key for x in (b >> 4, b & 15)]


def items_of(pairs):
    """{32-byte key: value bytes} as sorted model items"""
    return sorted((nibbles(k), bytes(v)) for k, v in pairs.items())


def _hp(nib, leaf):
    flag = (2 if leaf else 0) + (len(nib) & 1)
    out = [(flag << 4) | nib[0]] if len(nib) & 1 else [flag << 4]
    rest = nib[1:] if len(nib) & 1 else nib
    out += [(rest[i] << 4) | rest[i + 1] for i in range(0, len(rest), 2)]
    return bytes(out)


def _ref(raw):
    return synth.rlp_str(keccak(raw)) if len(raw) >= 32 else raw


def common_depth(items, depth):
    """the number of nibbles every item shares (at least `depth`)"""
    first, last = items[0][0], items[-1][0]
    cp = depth
    while first[cp] == last[cp]:
        cp += 1
    return cp


def split_children(items, depth):
    """the items below each of the 16 slots of a branch at `depth`"""
    kids = [[] for _ in range(16)]
    for it in items:
        kids[it[0][depth]].append(it)
    return kids


def node_rlp(items, depth):
    """RLP of the canonical trie node over items that share their first `depth` nibbles"""
    if len(items) == 1:
        nib, val = items[0]
        return synth.rlp_list([synth.rlp_str(_hp(nib[depth:], True)), synth.rlp_str(val)])
    cp = common_depth(items, depth)
    if cp > depth:
        return synth.rlp_list([synth.rlp_str(_hp(items[0][0][depth:cp], False)), _ref(node_rlp(items, cp))])
    kids = [_ref(node_rlp(sub, depth + 1)) if sub else b"\x80" for sub in split_children(items, depth)]
    return synth.rlp_list(kids + [b"\x80"])


def trie_root(pairs):
    """root of the trie of {32-byte key: value bytes}"""
    if not pairs:
        return EMPTY_TRIE_HASH
    return keccak(node_rlp(items_of(pairs), 0))


def subtrie_ref(items, depth):
    """What ppd_trie_subroot_sorted_leaves_dev returns for the part `items` below `depth` nibbles: the hash of its top
    node, or None when that node encodes to fewer than 32 bytes (the parent embeds such a node raw, so no 32-byte ref
    of it exists and the library must reject the part)."""
    raw = node_rlp(items, depth)
    return keccak(raw) if len(raw) >= 32 else None


Node = namedtuple("Node", "kind depth start_nibble nibble_count encoded_len n_children child_slots inline_child_slots")


def walk(items, depth=0):
    """Every node of the trie over `items` (top node first):
    (kind, depth, start_nibble, nibble_count, encoded_len, n_children, child_slots, inline_child_slots).
    kind is "leaf", "ext" or "branch"; start_nibble / nibble_count are the key nibbles the node spells (a branch spells
    none); encoded_len is the length of the node's RLP.  child_slots are a branch's occupied slots, inline_child_slots
    those whose child is embedded raw (shorter than 32 bytes); an extension has the one slot 0."""
    raw = node_rlp(items, depth)
    if len(items) == 1:
        yield Node("leaf", depth, depth, 64 - depth, len(raw), 0, (), ())
        return
    cp = common_depth(items, depth)
    if cp > depth:
        inline = len(node_rlp(items, cp)) < 32
        yield Node("ext", depth, depth, cp - depth, len(raw), 1, (0,), (0,) if inline else ())
        yield from walk(items, cp)
        return
    kids = split_children(items, depth)
    slots = tuple(n for n in range(16) if kids[n])
    inline = tuple(n for n in slots if len(node_rlp(kids[n], depth + 1)) < 32)
    yield Node("branch", depth, depth, 0, len(raw), len(slots), slots, inline)
    for n in slots:
        yield from walk(kids[n], depth + 1)


def payload_len(encoded_len):
    """the payload length of an RLP list of `encoded_len` bytes"""
    for hdr in (1, 2, 3, 4):
        p = encoded_len - hdr
        if (p < 56) == (hdr == 1) and (hdr == 1 or (p.bit_length() + 7) // 8 == hdr - 1):
            return p
    raise ValueError(encoded_len)
