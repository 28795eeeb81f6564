"""ctypes binding of libppd_b200.so (include/ppd_b200.h)."""
import ctypes
import weakref
import os
import subprocess

# Every block of a batch runs on its own CUDA stream; the device multiplexes streams onto CUDA_DEVICE_MAX_CONNECTIONS
# hardware queues (8 unless set, at most 32).  Must be in the environment before the process creates its CUDA context.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("PPD_LIB") or os.path.join(HERE, "libppd_b200.so")  # (PPD_LIB: a development build, csrc/Makefile "prof")
CSRC = os.path.join(HERE, "csrc")

STATUS_NAMES = {
    0: "OK",
    1: "MissingHeader",
    2: "InvalidOperator",
    3: "UnexpectedEndOfStream",
    4: "InvalidByteVector",
    5: "InvalidBytesForType",
    6: "InvalidWitnessFormat",
    7: "NonSingleEntryAfterProcessing",
    8: "IncorrectNumberOfNodesPrecedingBranch",
    9: "MissingExpectedNodesPrecedingBranch",
    10: "PrecedingNonNodeEntryFoundWhenProcessingRule",
    11: "KeyError",
    21: "AccountDecode",
    22: "MissingAccountStorageTrie",
    23: "NonExistentTrieEntry",
    24: "MissingKeysCreatingSubPartialTrie",
    25: "MissingWithdrawalAccount",
    40: "panic: incompatible header version",
    41: "panic: insert into hash node",
    42: "panic: H256::from_slice",
    43: "panic: receipt decode",
    44: "panic: pre-image account decode",
    45: "panic: unimplemented pre-image variant",
    46: "panic: key is a prefix of another key",
    47: "panic: U256::from_big_endian of more than 32 bytes",
    60: "bad flat input",
    61: "unresolved code hash",
    62: "bad argument",
    63: "unsorted keys",
    100: "CUDA error",
}


class PpdError(Exception):
    """A non-OK ppd_status.  Codes 1-11 are CompactParsingError variants, 21-25 TraceParsingError
    variants (decoding.rs:31-49), 40-47 places where the reference panics."""

    def __init__(self, code, msg=""):
        super().__init__(f"ppd status {code} ({STATUS_NAMES.get(code, '?')}): {msg}")
        self.code = code
        self.msg = msg  # ppd_last_error: for 21-25 the sentence is followed by "; key=value ..." (csrc/err_detail.h)

    def payload(self) -> dict:
        """The payload of a TraceParsingError variant (decoding.rs:31-49) as ppd_last_error spells it: hashed_addr / addr /
        amount / bytes as hex, trie_type as the reference's variant name."""
        if "; " not in self.msg:
            return {}
        return dict(w.split("=", 1) for w in self.msg.split("; ", 1)[1].split(" ") if "=" in w)


class PpdStats(ctypes.Structure):
    _fields_ = [
        ("nodes_hashed", ctypes.c_uint64),
        ("node_permutations", ctypes.c_uint64),
        ("key_hashes", ctypes.c_uint64),
        ("key_permutations", ctypes.c_uint64),
        ("node_bytes", ctypes.c_uint64),
        ("arena_nodes", ctypes.c_uint64),
        ("levels", ctypes.c_uint64),
        ("gpu_ms", ctypes.c_double),
        ("h2d_bytes", ctypes.c_double),
        ("d2h_bytes", ctypes.c_double),
        ("kernel_launches", ctypes.c_uint64),
        ("witnesses_on_gpu", ctypes.c_uint64),
        ("witness_instructions", ctypes.c_uint64),
        ("witness_bytes", ctypes.c_uint64),
        ("parse_gpu_ms", ctypes.c_double),
        ("level_launches", ctypes.c_uint64),
        ("marks_on_gpu", ctypes.c_uint64),
        ("txn_loops_on_gpu", ctypes.c_uint64),
        ("txn_gpu_ms", ctypes.c_double),
        ("dump_gpu_ms", ctypes.c_double),
        ("host_busy_ms", ctypes.c_double),
        ("host_wait_ms", ctypes.c_double),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


# void (*ppd_block_done_fn)(void* user, size_t index, int status, uint8_t* out, size_t out_len)
BLOCK_DONE_FN = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.POINTER(ctypes.c_uint8), ctypes.c_size_t)

EXPORTS = [
    "ppd_ctx_create",
    "ppd_ctx_destroy",
    "ppd_last_error",
    "ppd_last_stats",
    "ppd_free",
    "ppd_alloc_pinned",
    "ppd_keccak256_batch",
    "ppd_compact_decode",
    "ppd_block_decode",
    "ppd_blocks_decode_batch",
    "ppd_trie_root_sorted_leaves",
    "ppd_trie_root_sorted_leaves_dev",
    "ppd_trie_subroot_sorted_leaves_dev",
    "ppd_trie_root_from_children",
    "ppd_blocks_decode_stream",
    "ppd_replay_last",
    "ppd_replay_lanes",
    "ppd_replay_last_hashing",
    "ppd_replay_last_parse",
    "ppd_microbench",
    "ppd_direct_to_compact",
    "ppd_trie_root_leaves",
    "ppd_trie_root_leaves_dev",
]

LEAVES_HASH_KEYS = 1  # PPD_LEAVES_HASH_KEYS: key i is keccak256 of the given key bytes


def build_extension(verbose=False):
    """Compile every CUDA source for sm_100a into libppd_b200.so, in-tree (nvcc cross-compiles without a GPU)."""
    res = subprocess.run(["make", "-C", CSRC], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("building libppd_b200.so failed:\n" + res.stdout + res.stderr)
    if verbose:
        print(res.stdout)
    return SO_PATH


class PpdLibrary:
    def __init__(self, path=SO_PATH):
        if not os.path.exists(path):
            raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (there is no CPU fallback)")
        L = ctypes.CDLL(path)
        self.L = L
        u8pp = ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8))
        szp = ctypes.POINTER(ctypes.c_size_t)
        L.ppd_ctx_create.argtypes = [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]
        L.ppd_ctx_destroy.argtypes = [ctypes.c_void_p]
        L.ppd_last_error.argtypes = [ctypes.c_void_p]
        L.ppd_last_error.restype = ctypes.c_char_p
        L.ppd_last_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(PpdStats)]
        L.ppd_free.argtypes = [ctypes.c_void_p]
        L.ppd_alloc_pinned.argtypes = [ctypes.c_size_t]
        L.ppd_alloc_pinned.restype = ctypes.c_void_p
        L.ppd_keccak256_batch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]
        L.ppd_compact_decode.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, u8pp, szp]
        L.ppd_block_decode.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, u8pp, szp]
        L.ppd_blocks_decode_batch.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.ppd_trie_root_sorted_leaves.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p]
        L.ppd_replay_last.argtypes = [ctypes.c_void_p, ctypes.c_uint, ctypes.POINTER(ctypes.c_double)]
        L.ppd_blocks_decode_stream.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, BLOCK_DONE_FN, ctypes.c_void_p]
        L.ppd_replay_lanes.argtypes = [ctypes.c_void_p]
        L.ppd_replay_lanes.restype = ctypes.c_size_t
        L.ppd_replay_last_hashing.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
        L.ppd_replay_last_parse.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
        L.ppd_microbench.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint32)]
        L.ppd_trie_root_sorted_leaves_dev.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_char_p]
        L.ppd_trie_subroot_sorted_leaves_dev.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_char_p]
        L.ppd_trie_root_from_children.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p]

        L.ppd_direct_to_compact.argtypes = [ctypes.c_void_p, ctypes.c_size_t, u8pp, szp]
        L.ppd_trie_root_leaves.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_char_p]
        L.ppd_trie_root_leaves_dev.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_char_p]

    def exported(self):
        return [name for name in EXPORTS if hasattr(self.L, name)]

    def direct_to_compact(self, direct: bytes) -> bytes:
        """ppd_direct_to_compact: a DirectPreImage payload (FlatBlock pre_image_kind 2) as the TrieCompact witness of the
        same tries.  Host only: needs no context and no device."""
        out, n = ctypes.POINTER(ctypes.c_uint8)(), ctypes.c_size_t()
        buf = ctypes.create_string_buffer(bytes(direct), len(direct)) if len(direct) else ctypes.create_string_buffer(1)
        rc = self.L.ppd_direct_to_compact(buf, len(direct), ctypes.byref(out), ctypes.byref(n))
        if rc != 0:
            raise PpdError(rc, "ppd_direct_to_compact")
        try:
            return ctypes.string_at(out, n.value)
        finally:
            self.L.ppd_free(out)


class OwnedBuffer:
    """A buffer allocated by the library (released with ppd_free), exposed without copying."""

    def __init__(self, lib, ptr, n):
        self._lib, self._ptr, self.nbytes = lib, ptr, n
        self.view = memoryview((ctypes.c_uint8 * n).from_address(ctypes.addressof(ptr.contents))).cast("B") if n else memoryview(b"")

    def close(self):
        if self._ptr is not None:
            self.view = None
            self._lib.L.ppd_free(self._ptr)
            self._ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Context:
    """One ppd_ctx: a stream plus reusable HBM buffers on one CUDA device.  Not thread-safe."""

    def __init__(self, device=0, lib=None):
        self.lib = lib or load_library()
        self.h = ctypes.c_void_p()
        rc = self.lib.L.ppd_ctx_create(device, ctypes.byref(self.h))
        if rc != 0:
            raise PpdError(rc, "ppd_ctx_create failed: no usable CUDA device (there is no CPU fallback)")

    def close(self):
        if self.h:
            self.lib.L.ppd_ctx_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PpdError(rc, self.lib.L.ppd_last_error(self.h).decode(errors="replace"))

    def stats(self):
        s = PpdStats()
        self.lib.L.ppd_last_stats(self.h, ctypes.byref(s))
        return s.as_dict()

    def _take(self, out, n):
        data = ctypes.string_at(out, n.value)
        self.lib.L.ppd_free(out)
        return data

    def keccak256_batch(self, data, offsets):
        import numpy as np

        data = np.ascontiguousarray(data, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        n = len(offsets) - 1
        out = np.empty((n, 32), dtype=np.uint8)
        self._check(self.lib.L.ppd_keccak256_batch(self.h, data.ctypes.data, offsets.ctypes.data, n, out.ctypes.data))
        return out

    def pinned_copy(self, data):
        """`data` (bytes or a uint8 numpy array) copied into a page-locked buffer from the library's pool
        (ppd_alloc_pinned); returns a uint8 numpy array over it.  The buffer goes back to the pool when the
        array (and every view of it) is garbage collected."""
        import numpy as np

        src = np.frombuffer(data, dtype=np.uint8) if isinstance(data, (bytes, bytearray, memoryview)) else np.ascontiguousarray(data, dtype=np.uint8)
        n = int(src.nbytes)
        p = self.lib.L.ppd_alloc_pinned(n)
        if not p:
            raise MemoryError("ppd_alloc_pinned")
        raw = (ctypes.c_uint8 * max(n, 1)).from_address(p)
        arr = np.frombuffer(raw, dtype=np.uint8, count=n)
        arr[:] = src
        lib = self.lib
        weakref.finalize(raw, lib.L.ppd_free, ctypes.c_void_p(p))
        return arr

    def compact_decode(self, witness: bytes) -> bytes:
        out, n = ctypes.POINTER(ctypes.c_uint8)(), ctypes.c_size_t()
        buf = ctypes.create_string_buffer(bytes(witness), len(witness)) if len(witness) else ctypes.create_string_buffer(1)
        self._check(self.lib.L.ppd_compact_decode(self.h, buf, len(witness), ctypes.byref(out), ctypes.byref(n)))
        return self._take(out, n)

    def block_decode(self, flat: bytes) -> bytes:
        with self.block_decode_view(flat) as v:
            return bytes(v.view)

    def block_decode_view(self, flat) -> "OwnedBuffer":
        """ppd_block_decode without any copy on the Python side: `flat` (bytes or a C-contiguous uint8
        numpy array) is passed by address and the library-allocated IrDump is returned as an
        OwnedBuffer (memoryview + ppd_free on close)."""
        out, n = ctypes.POINTER(ctypes.c_uint8)(), ctypes.c_size_t()
        if isinstance(flat, (bytes, bytearray)):
            ptr, ln = ctypes.cast(ctypes.c_char_p(bytes(flat) if isinstance(flat, bytearray) else flat), ctypes.c_void_p), len(flat)
        else:
            ptr, ln = ctypes.c_void_p(flat.ctypes.data), flat.nbytes
        self._check(self.lib.L.ppd_block_decode(self.h, ptr, ln, ctypes.byref(out), ctypes.byref(n)))
        return OwnedBuffer(self.lib, out, n.value)

    def blocks_decode_batch(self, flats):
        res = []
        for v in self.blocks_decode_batch_view(flats):
            if isinstance(v, PpdError):
                res.append(v)
            else:
                with v:
                    res.append(bytes(v.view))
        return res

    def blocks_decode_batch_view(self, flats):
        """ppd_blocks_decode_batch without copies on the Python side: inputs by address, outputs as
        OwnedBuffer (or PpdError for a block that failed on its own)."""
        n = len(flats)
        keep = [bytes(f) if isinstance(f, bytearray) else f for f in flats]
        addr = [ctypes.cast(ctypes.c_char_p(f), ctypes.c_void_p).value if isinstance(f, bytes) else f.ctypes.data for f in keep]
        ptrs = (ctypes.c_void_p * n)(*addr)
        lens = (ctypes.c_size_t * n)(*[len(f) if isinstance(f, bytes) else f.nbytes for f in keep])
        outs = (ctypes.POINTER(ctypes.c_uint8) * n)()
        out_lens = (ctypes.c_size_t * n)()
        statuses = (ctypes.c_int * n)()
        self._check(self.lib.L.ppd_blocks_decode_batch(self.h, ptrs, lens, n, outs, out_lens, statuses))
        res = []
        for i in range(n):
            if statuses[i] == 0:
                res.append(OwnedBuffer(self.lib, ctypes.cast(outs[i], ctypes.POINTER(ctypes.c_uint8)), out_lens[i]))
            else:
                res.append(PpdError(statuses[i], "block %d" % i))
        return res

    def blocks_decode_stream(self, flats, on_done):
        """ppd_blocks_decode_stream: on_done(index, result) is called as each block finishes (from the library's host
        threads, in completion order); result is an OwnedBuffer (close it when done) or a PpdError."""
        n = len(flats)
        keep = [bytes(f) if isinstance(f, bytearray) else f for f in flats]
        addr = [ctypes.cast(ctypes.c_char_p(f), ctypes.c_void_p).value if isinstance(f, bytes) else f.ctypes.data for f in keep]
        ptrs = (ctypes.c_void_p * n)(*addr)
        lens = (ctypes.c_size_t * n)(*[len(f) if isinstance(f, bytes) else f.nbytes for f in keep])
        failure = []

        def tramp(_user, index, status, out, out_len):
            try:
                on_done(index, OwnedBuffer(self.lib, out, out_len) if status == 0 else PpdError(status, "block %d" % index))
            except BaseException as e:  # noqa: BLE001 — raised again on the calling thread
                failure.append(e)

        cb = BLOCK_DONE_FN(tramp)
        self._check(self.lib.L.ppd_blocks_decode_stream(self.h, ptrs, lens, n, cb, None))
        if failure:
            raise failure[0]

    REPLAY_PARSE, REPLAY_HASH, REPLAY_TXN, REPLAY_DUMP, REPLAY_ALL = 1, 2, 4, 8, 15

    def replay_last(self, what=15) -> float:
        """Device time (ms) of the selected stages of the last decode call, re-run on what is resident in HBM."""
        ms = ctypes.c_double()
        self._check(self.lib.L.ppd_replay_last(self.h, what, ctypes.byref(ms)))
        return ms.value

    def replay_lanes(self) -> int:
        """How many lanes (= resident blocks) replay_last covers."""
        return int(self.lib.L.ppd_replay_lanes(self.h))

    def replay_last_hashing(self) -> float:
        ms = ctypes.c_double()
        self._check(self.lib.L.ppd_replay_last_hashing(self.h, ctypes.byref(ms)))
        return ms.value

    def replay_last_parse(self) -> float:
        ms = ctypes.c_double()
        self._check(self.lib.L.ppd_replay_last_parse(self.h, ctypes.byref(ms)))
        return ms.value

    def microbench(self, variant, blocks_per_sm=8, iters=2000):
        ms, units = ctypes.c_double(), ctypes.c_double()
        dig = (ctypes.c_uint32 * 2)()
        self._check(self.lib.L.ppd_microbench(self.h, variant, blocks_per_sm, iters, ctypes.byref(ms), ctypes.byref(units), dig))
        return ms.value, units.value, (dig[0], dig[1])

    def trie_root_sorted_leaves(self, keys, val_off, vals) -> bytes:
        import numpy as np

        keys = np.ascontiguousarray(keys, dtype=np.uint8)
        val_off = np.ascontiguousarray(val_off, dtype=np.uint64)
        vals = np.ascontiguousarray(vals, dtype=np.uint8)
        out = ctypes.create_string_buffer(32)
        self._check(self.lib.L.ppd_trie_root_sorted_leaves(self.h, keys.ctypes.data, val_off.ctypes.data, vals.ctypes.data, len(val_off) - 1, out))
        return out.raw

    def trie_root_sorted_leaves_dev(self, d_keys_ptr, d_val_off_ptr, d_vals_ptr, n, vals_bytes) -> bytes:
        out = ctypes.create_string_buffer(32)
        self._check(self.lib.L.ppd_trie_root_sorted_leaves_dev(self.h, d_keys_ptr, d_val_off_ptr, d_vals_ptr, n, vals_bytes, out))
        return out.raw


    def trie_root_leaves(self, keys, val_off, vals, hash_keys=False) -> bytes:
        """Root of the trie that inserting the leaves in order gives: keys in any order, a repeated key keeps its last
        value.  keys: uint8 [n, key_len] (key_len 32, or 1..135 with hash_keys: the key is then keccak256 of the row)."""
        import numpy as np

        keys = np.ascontiguousarray(keys, dtype=np.uint8)
        val_off = np.ascontiguousarray(val_off, dtype=np.uint64)
        vals = np.ascontiguousarray(vals, dtype=np.uint8)
        if keys.ndim != 2 or keys.shape[0] != len(val_off) - 1:
            raise ValueError("keys must be [n, key_len] with n = len(val_off) - 1")
        out = ctypes.create_string_buffer(32)
        flags = LEAVES_HASH_KEYS if hash_keys else 0
        self._check(self.lib.L.ppd_trie_root_leaves(self.h, keys.ctypes.data, keys.shape[1], flags, val_off.ctypes.data, vals.ctypes.data, keys.shape[0], out))
        return out.raw

    def trie_root_leaves_dev(self, d_keys_ptr, key_len, d_val_off_ptr, d_vals_ptr, n, vals_bytes, hash_keys=False, flags=None) -> bytes:
        """trie_root_leaves on device buffers (e.g. torch tensors' data_ptr()), which must be complete when it is called: the
        library reads them on a stream of its own (torch.cuda.synchronize() first).  `flags` overrides hash_keys when given."""
        out = ctypes.create_string_buffer(32)
        if flags is None:
            flags = LEAVES_HASH_KEYS if hash_keys else 0
        self._check(self.lib.L.ppd_trie_root_leaves_dev(self.h, d_keys_ptr, key_len, flags, d_val_off_ptr, d_vals_ptr, n, vals_bytes, out))
        return out.raw

    def trie_subroot_sorted_leaves_dev(self, d_keys_ptr, d_val_off_ptr, d_vals_ptr, n, vals_bytes, base_depth) -> bytes:
        """The ref of the sub-trie over n sorted leaves that share their first base_depth nibbles (device pointers)."""
        out = ctypes.create_string_buffer(32)
        self._check(self.lib.L.ppd_trie_subroot_sorted_leaves_dev(self.h, d_keys_ptr, d_val_off_ptr, d_vals_ptr, n, vals_bytes, base_depth, out))
        return out.raw

    def trie_root_from_children(self, child_hashes, mask) -> bytes:
        """Root of the branch whose child i (bit i of mask) has the 32-byte ref child_hashes[32 * i : 32 * i + 32]."""
        out = ctypes.create_string_buffer(32)
        buf = bytes(child_hashes).ljust(512, b"\0")
        self._check(self.lib.L.ppd_trie_root_from_children(self.h, buf, mask, out))
        return out.raw


_lib = None


def load_library():
    global _lib
    if _lib is None:
        _lib = PpdLibrary()
    return _lib
