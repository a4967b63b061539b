"""sourmash_rust_b200 -- Python binding (ctypes) of this build's libsourmash.so.

The product is the C ABI of include/sourmash.h + include/sourmash_b200.h; this module is the thin
host-side mirror used by the tests and the benchmark, with the reference crate's names
(KmerMinHash::new / add_sequence / add_hash / merge / compare / count_common ..., src/lib.rs:141-513;
Signature, src/lib.rs:546-675).  Every call goes through the C ABI and runs on the GPU; there is
no Python or CPU implementation behind it -- if the shared library is missing or no CUDA device is
usable, calls raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SMB200_LIB") or os.path.join(_HERE, "libsourmash.so")  # override: kernel A/B runs

u64, u32, i32, usz, vp, cb = C.c_uint64, C.c_uint32, C.c_int32, C.c_size_t, C.c_void_p, C.c_bool
p_u64 = C.POINTER(C.c_uint64)


class SourmashStr(C.Structure):
    _fields_ = [("data", C.POINTER(C.c_char)), ("len", C.c_size_t), ("owned", C.c_bool)]


# name -> (restype, argtypes); exactly the declarations of include/sourmash.h ...
REFERENCE_ABI = {
    "hash_murmur": (u64, [C.c_char_p, u64]),
    "kmerminhash_new": (vp, [u32, u32, cb, u64, u64, cb]),
    "kmerminhash_free": (None, [vp]),
    "kmerminhash_add_sequence": (None, [vp, C.c_char_p, cb]),
    "kmerminhash_add_hash": (None, [vp, u64]),
    "kmerminhash_add_word": (None, [vp, C.c_char_p]),
    "kmerminhash_add_from": (None, [vp, vp]),
    "kmerminhash_mins_push": (None, [vp, u64]),
    "kmerminhash_abunds_push": (None, [vp, u64]),
    "kmerminhash_merge": (None, [vp, vp]),
    "kmerminhash_compare": (C.c_double, [vp, vp]),
    "kmerminhash_count_common": (u64, [vp, vp]),
    "kmerminhash_intersection": (u64, [vp, vp]),
    "kmerminhash_get_mins": (p_u64, [vp]),
    "kmerminhash_get_abunds": (p_u64, [vp]),
    "kmerminhash_get_mins_size": (usz, [vp]),
    "kmerminhash_get_abunds_size": (usz, [vp]),
    "kmerminhash_get_min_idx": (u64, [vp, u64]),
    "kmerminhash_get_abund_idx": (u64, [vp, u64]),
    "kmerminhash_is_protein": (cb, [vp]),
    "kmerminhash_seed": (u64, [vp]),
    "kmerminhash_track_abundance": (cb, [vp]),
    "kmerminhash_num": (u32, [vp]),
    "kmerminhash_ksize": (u32, [vp]),
    "kmerminhash_max_hash": (u64, [vp]),
    "signature_new": (vp, []),
    "signature_free": (None, [vp]),
    "signature_set_name": (None, [vp, C.c_char_p]),
    "signature_set_filename": (None, [vp, C.c_char_p]),
    "signature_push_mh": (None, [vp, vp]),
    "signature_set_mh": (None, [vp, vp]),
    "signature_get_name": (SourmashStr, [vp]),
    "signature_get_filename": (SourmashStr, [vp]),
    "signature_get_license": (SourmashStr, [vp]),
    "signature_first_mh": (vp, [vp]),
    "signature_get_mhs": (C.POINTER(vp), [vp, C.POINTER(usz)]),
    "signature_eq": (cb, [vp, vp]),
    "signature_save_json": (SourmashStr, [vp]),
    "signatures_save_buffer": (SourmashStr, [C.POINTER(vp), usz]),
    "signatures_load_path": (C.POINTER(vp), [C.c_char_p, cb, usz, C.c_char_p, C.POINTER(usz)]),
    "signatures_load_buffer": (C.POINTER(vp), [C.c_char_p, usz, cb, usz, C.c_char_p, C.POINTER(usz)]),
    "sourmash_init": (None, []),
    "sourmash_err_clear": (None, []),
    "sourmash_err_get_last_code": (u32, []),
    "sourmash_err_get_last_message": (SourmashStr, []),
    "sourmash_err_get_backtrace": (SourmashStr, []),
    "sourmash_str_free": (None, [C.POINTER(SourmashStr)]),
    "sourmash_str_from_cstr": (SourmashStr, [C.c_char_p]),
}
# ... and of include/sourmash_b200.h
EXTENSION_ABI = {
    "smgpu_set_device": (None, [i32]),
    "smgpu_device": (i32, [C.POINTER(i32)]),
    "smgpu_launch_count": (u64, []),
    "smgpu_stream": (u64, []),
    "smgpu_profile_enable": (None, [cb]),
    "smgpu_profile_read": (None, [i32, C.POINTER(C.c_double), C.POINTER(u64), cb]),
    "smgpu_int_peak": (C.c_double, [i32, i32, i32]),
    "smgpu_fuse_multi_k": (None, [C.c_bool]),
    "smgpu_alloc_pinned": (vp, [usz]),
    "smgpu_free_pinned": (None, [vp]),
    "kmerminhash_slice_free": (None, [p_u64]),
    "kmerminhash_jaccard": (C.c_double, [vp, vp]),
    "kmerminhash_containment": (C.c_double, [vp, vp]),
    "kmerminhash_intersection_hashes": (p_u64, [vp, vp, C.POINTER(usz), C.POINTER(u64)]),
    "kmerminhash_add_sequences": (None, [C.POINTER(vp), usz, vp, vp, u64, cb, cb]),
    "kmerminhash_add_reads": (None, [C.POINTER(vp), usz, vp, u64, u32, cb, cb]),
    "kmerminhash_add_reads_2bit": (None, [C.POINTER(vp), usz, vp, u64, u32, cb]),
    "kmerminhash_set_mins": (None, [vp, vp, usz, vp, usz]),
    "kmerminhash_copy_mins": (usz, [vp, vp, vp, cb]),
    "kmerminhash_md5sum": (SourmashStr, [vp]),
    "smgpu_collection_new": (vp, []),
    "smgpu_collection_free": (None, [vp]),
    "smgpu_collection_push": (None, [vp, vp]),
    "smgpu_collection_push_signatures": (None, [vp, vp, usz]),
    "smgpu_collection_from_csr": (vp, [vp, vp, u64, u32, u32, u64, u64, cb]),
    "smgpu_sketch_collection": (vp, [vp, vp, u64, u32, u32, u64, u64, cb]),
    "smgpu_collection_len": (u64, [vp]),
    "smgpu_collection_copy": (u64, [vp, vp, vp]),
    "smgpu_collection_csr": (u64, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "smgpu_compare_matrix": (None, [vp, u64, u64, vp, u64, u64, i32, vp, vp, vp, u64, cb]),
    "smgpu_scaffold_pairs": (u64, [vp, vp, vp]),
    "smgpu_compare_path": (None, [i32]),
    "smgpu_find_path": (None, [i32]),
    "smgpu_linear_find": (u64, [vp, vp, i32, C.c_double, vp, vp, u64]),
    "smgpu_comm_unique_id": (None, [vp]),
    "smgpu_comm_init": (None, [vp, i32, i32]),
    "smgpu_comm_destroy": (None, []),
    "smgpu_comm_rank": (i32, []),
    "smgpu_comm_world": (i32, []),
    "smgpu_comm_nccl_version": (i32, []),
    "smgpu_collection_allgather": (vp, [vp]),
    "smgpu_compare_matrix_allgather": (vp, [vp, i32, vp, vp, vp, u64, cb]),
    "smgpu_comm_allmerge": (None, [vp]),
    "smgpu_linear_find_sharded": (u64, [vp, vp, i32, C.c_double, vp, vp, u64]),
    "smgpu_nodegraph_new": (vp, [vp, usz, u64]),
    "smgpu_nodegraph_free": (None, [vp]),
    "smgpu_nodegraph_from_buffer": (vp, [C.c_char_p, usz]),
    "smgpu_nodegraph_save": (usz, [vp, vp, usz]),
    "smgpu_nodegraph_count_many": (u64, [vp, vp, u64, vp, cb]),
    "smgpu_nodegraph_get_many": (u64, [vp, vp, u64, vp, cb]),
    "smgpu_nodegraph_matches": (u64, [vp, vp]),
    "smgpu_nodegraph_update": (None, [vp, vp]),
    "smgpu_nodegraph_similarity": (C.c_double, [vp, vp]),
    "smgpu_nodegraph_containment": (C.c_double, [vp, vp]),
    "smgpu_nodegraph_tablesizes": (usz, [vp, vp, usz]),
    "smgpu_nodegraph_ksize": (u64, [vp]),
    "smgpu_nodegraph_n_occupied_bins": (u64, [vp]),
    "smgpu_nodegraph_unique_kmers": (u64, [vp]),
    "smgpu_sbt_find": (u64, [u32, vp, vp, vp, u64, vp, vp, vp, i32, C.c_double, vp, vp, u64]),
}

_lib = None


def lib():
    """The loaded C-ABI library (raises if it has not been built: see build.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s is missing: run `python -m sourmash_rust_b200.build` (there is no fallback path)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for table in (REFERENCE_ABI, EXTENSION_ABI):
            for name, (res, args) in table.items():
                f = getattr(L, name)
                f.restype, f.argtypes = res, args
        _lib = L
    return _lib


class SourmashError(Exception):
    def __init__(self, code, message):
        super().__init__("[%d] %s" % (code, message))
        self.code = code
        self.message = message


def _take_str(s: SourmashStr) -> bytes:
    out = C.string_at(s.data, s.len) if s.len else b""
    lib().sourmash_str_free(C.byref(s))
    return out


def _check():
    """The caller protocol of the reference ABI: read the thread-local error after a call."""
    L = lib()
    code = L.sourmash_err_get_last_code()
    if code:
        msg = _take_str(L.sourmash_err_get_last_message()).decode("utf-8", "replace")
        L.sourmash_err_clear()
        raise SourmashError(code, msg)


def _call(name, *args):
    L = lib()
    L.sourmash_err_clear()
    r = getattr(L, name)(*args)
    _check()
    return r


def hash_murmur(kmer: bytes, seed: int = 42) -> int:
    return _call("hash_murmur", kmer, seed)


def set_device(device: int):
    _call("smgpu_set_device", device)


def device_info():
    sm = i32(0)
    dev = _call("smgpu_device", C.byref(sm))
    return dev, sm.value


def launch_count() -> int:
    return lib().smgpu_launch_count()


def stream_handle() -> int:
    return _call("smgpu_stream")


def profile_enable(on=True):
    lib().smgpu_profile_enable(on)


PROFILE_KINDS = {"sketch_k21": 0, "sketch_k31": 1, "sketch_k51": 2, "sketch_other": 3, "compare": 4, "join_sort": 5,
                 "sketch_multi": 6, "find_stream": 7, "compare_walk": 8, "compare_probe": 9, "compare_fill": 10}


def compare_path(path="auto"):
    """'auto' | 'dense' | 'sparse' (smgpu_compare_path)"""
    lib().smgpu_compare_path({"auto": 0, "dense": 1, "sparse": 2}[path])


def find_path(path="auto"):
    """'auto' | 'join' | 'stream' | 'stream_small_spill' (smgpu_find_path)"""
    lib().smgpu_find_path({"auto": 0, "join": 1, "stream": 2, "stream_small_spill": 3}[path])


def fuse_multi_k(on=True):
    """Fused multi-k launches in batch sketching on/off (smgpu_fuse_multi_k)."""
    lib().smgpu_fuse_multi_k(bool(on))


def profile_read(kind, reset=False):
    ms, n = C.c_double(0), u64(0)
    _call("smgpu_profile_read", PROFILE_KINDS[kind], C.byref(ms), C.byref(n), reset)
    return ms.value, n.value


def int_peak(mode=2, iters=4096, blocks=148 * 8):
    return _call("smgpu_int_peak", mode, iters, blocks)


def _vp(x):
    """Host numpy array / bytes, or a raw integer device pointer -> c_void_p."""
    if x is None:
        return None
    if isinstance(x, int):
        return C.c_void_p(x)
    if isinstance(x, np.ndarray):
        return C.c_void_p(x.ctypes.data)
    if isinstance(x, (bytes, bytearray)):
        return C.cast(C.c_char_p(bytes(x)), C.c_void_p)
    raise TypeError(type(x))


class KmerMinHash:
    """KmerMinHash::new(num, ksize, is_protein, seed, max_hash, track_abundance) (lib.rs:142-149)."""

    def __init__(self, num, ksize, is_protein=False, seed=42, max_hash=0, track_abundance=False, _ptr=None):
        self._p = _ptr if _ptr is not None else _call("kmerminhash_new", num, ksize, is_protein, seed, max_hash,
                                                      track_abundance)

    def __del__(self):
        p, self._p = getattr(self, "_p", None), None
        if p and _lib is not None:
            _lib.kmerminhash_free(p)

    # --- scalar getters -------------------------------------------------------------------
    num = property(lambda s: _call("kmerminhash_num", s._p))
    ksize = property(lambda s: _call("kmerminhash_ksize", s._p))
    seed = property(lambda s: _call("kmerminhash_seed", s._p))
    max_hash = property(lambda s: _call("kmerminhash_max_hash", s._p))
    is_protein = property(lambda s: _call("kmerminhash_is_protein", s._p))

    def track_abundance(self):
        return _call("kmerminhash_track_abundance", self._p)

    # --- ingest -----------------------------------------------------------------------------
    def add_sequence(self, seq: bytes, force=False):
        if b"\0" in seq:
            raise ValueError("NUL inside a sequence (the C ABI takes NUL-terminated strings)")
        _call("kmerminhash_add_sequence", self._p, seq, force)

    def add_hash(self, h):
        _call("kmerminhash_add_hash", self._p, h)

    def add_word(self, w: bytes):
        _call("kmerminhash_add_word", self._p, w)

    def add_from(self, other):
        _call("kmerminhash_add_from", self._p, other._p)

    def add_many(self, hashes):
        for h in hashes:
            self.add_hash(int(h))

    def mins_push(self, v):
        _call("kmerminhash_mins_push", self._p, v)

    def abunds_push(self, v):
        _call("kmerminhash_abunds_push", self._p, v)

    def set_mins(self, mins, abunds=None):
        m = np.ascontiguousarray(mins, dtype=np.uint64)
        a = None if abunds is None else np.ascontiguousarray(abunds, dtype=np.uint64)
        _call("kmerminhash_set_mins", self._p, _vp(m), m.size, _vp(a), 0 if a is None else a.size)

    def add_reads(self, buf, n_reads, read_len, force=True, on_device=False):
        add_reads([self], buf, n_reads, read_len, force, on_device)

    def add_sequences(self, buf, offsets, force=True, on_device=False, n_seqs=None):
        add_sequences([self], buf, offsets, force, on_device, n_seqs)

    # --- combine / compare ----------------------------------------------------------------
    def merge(self, other):
        _call("kmerminhash_merge", self._p, other._p)

    def compare(self, other):
        return _call("kmerminhash_compare", self._p, other._p)

    def jaccard(self, other):
        """north_star's name for `compare` (lib.rs:501-508), through its own C symbol."""
        return _call("kmerminhash_jaccard", self._p, other._p)

    def intersection(self, other):
        """KmerMinHash::intersection (lib.rs:438-468): (common hashes within combined, |combined|)."""
        n, size = usz(0), u64(0)
        p = _call("kmerminhash_intersection_hashes", self._p, other._p, C.byref(n), C.byref(size))
        out = np.ctypeslib.as_array(p, shape=(n.value,)).copy() if n.value else np.zeros(0, dtype=np.uint64)
        lib().kmerminhash_slice_free(p)
        return out, size.value

    def count_common(self, other):
        return _call("kmerminhash_count_common", self._p, other._p)

    def intersection_union_size(self, other):
        """kmerminhash_intersection: the (truncated) union size (ffi.rs:292-309)."""
        return _call("kmerminhash_intersection", self._p, other._p)

    def containment(self, query):
        """Leaf<Signature>::containment with self as the node: |self n query| / |self| (index.rs:146-160)."""
        return _call("kmerminhash_containment", self._p, query._p)

    similarity = compare  # Leaf<Signature>::similarity (index.rs:131-144)

    # --- read-out ---------------------------------------------------------------------------
    def size(self):
        return _call("kmerminhash_get_mins_size", self._p)

    def mins_np(self):
        n = self.size()
        out = np.zeros(n, dtype=np.uint64)
        if n:
            _call("kmerminhash_copy_mins", self._p, _vp(out), None, False)
        return out

    def abunds_np(self):
        if not self.track_abundance():
            return None
        n = _call("kmerminhash_get_abunds_size", self._p)
        if n == 0:
            return np.zeros(0, dtype=np.uint64)
        p = _call("kmerminhash_get_abunds", self._p)
        out = np.ctypeslib.as_array(p, shape=(n,)).copy()
        lib().kmerminhash_slice_free(p)
        return out

    @property
    def mins(self):
        n = self.size()
        p = _call("kmerminhash_get_mins", self._p)
        out = [p[i] for i in range(n)]
        lib().kmerminhash_slice_free(p)
        return out

    @property
    def abunds(self):
        a = self.abunds_np()
        return None if a is None else [int(x) for x in a]

    def get_min_idx(self, i):
        return _call("kmerminhash_get_min_idx", self._p, i)

    def get_abund_idx(self, i):
        return _call("kmerminhash_get_abund_idx", self._p, i)

    def md5sum(self):
        return _take_str(_call("kmerminhash_md5sum", self._p)).decode()


def _handles(mhs):
    return (vp * len(mhs))(*[m._p for m in mhs])


def add_reads(mhs, buf, n_reads, read_len, force=True, on_device=False):
    """kmerminhash_add_reads: every read added to every sketch of `mhs` in one pass."""
    keep = buf if (on_device or isinstance(buf, (int, np.ndarray))) else bytes(buf)  # int = raw pointer
    _call("kmerminhash_add_reads", _handles(mhs), len(mhs), _vp(keep), n_reads, read_len, force, on_device)


def add_reads_2bit(mhs, packed, n_reads, read_len, on_device=False):
    """kmerminhash_add_reads_2bit (NOT a reference format): reads stored 2 bits per base, see include/sourmash_b200.h."""
    keep = packed if (on_device or isinstance(packed, (int, np.ndarray))) else bytes(packed)
    _call("kmerminhash_add_reads_2bit", _handles(mhs), len(mhs), _vp(keep), n_reads, read_len, on_device)


def pack_2bit(reads: np.ndarray, read_len: int) -> np.ndarray:
    """Host helper for tests / benches: ASCII reads (n x read_len uint8, ACGT only) -> the 2-bit form above."""
    r = np.ascontiguousarray(reads, dtype=np.uint8).reshape(-1, read_len)
    lut = np.zeros(256, dtype=np.uint8)
    lut[list(b"ACGT")] = [0, 1, 2, 3]
    codes = lut[r]
    pad = (-read_len) % 4
    if pad:
        codes = np.concatenate([codes, np.zeros((codes.shape[0], pad), dtype=np.uint8)], axis=1)
    q = codes.reshape(codes.shape[0], -1, 4)
    return np.ascontiguousarray(q[:, :, 0] | (q[:, :, 1] << 2) | (q[:, :, 2] << 4) | (q[:, :, 3] << 6))


def add_sequences(mhs, buf, offsets, force=True, on_device=False, n_seqs=None):
    """kmerminhash_add_sequences: sequence s = buf[offsets[s]:offsets[s+1]]."""
    if on_device:
        keep_b, keep_o = buf, offsets
        assert n_seqs is not None
    else:
        keep_b = buf if isinstance(buf, (int, np.ndarray)) else bytes(buf)
        keep_o = np.ascontiguousarray(offsets, dtype=np.uint64)
        n_seqs = keep_o.size - 1
    _call("kmerminhash_add_sequences", _handles(mhs), len(mhs), _vp(keep_b), _vp(keep_o), n_seqs, force, on_device)


_feed = None


def feed_reads(mh_groups, reads, n_reads, stride, force=False, warm_reads=0, flush=True):
    """The reference's calling pattern for a read set, timed natively: a C loop (host/feed_reads.c) calls
    kmerminhash_add_sequence once per read and per sketch.  `reads` (numpy array or raw host pointer) holds n_reads
    NUL-terminated strings, one every `stride` bytes; mh_groups is a list (one entry per host thread) of equally
    long lists of sketches -- thread t feeds its sketches with its contiguous share of the reads, the first
    `warm_reads` of them untimed.  With `flush` the timed region ends with kmerminhash_get_mins_size on every
    sketch, i.e. with all deferred work done.  Returns the timed region's wall time in seconds."""
    global _feed
    if _feed is None:
        path = os.path.join(_HERE, "libfeedreads.so")
        if not os.path.exists(path):
            raise RuntimeError("%s is missing: run `python -m sourmash_rust_b200.build`" % path)
        F = C.CDLL(path)
        F.feed_reads_mt.restype = u64
        F.feed_reads_mt.argtypes = [vp, vp, C.POINTER(vp), C.c_int, C.c_int, vp, u64, u64, cb, u64]
        _feed = F
    n_mhs = len(mh_groups[0])
    assert all(len(g) == n_mhs for g in mh_groups)
    flat = (vp * (n_mhs * len(mh_groups)))(*[m._p for g in mh_groups for m in g])
    fn = C.cast(lib().kmerminhash_add_sequence, vp)
    lib().sourmash_err_clear()
    size_fn = C.cast(lib().kmerminhash_get_mins_size, vp) if flush else None
    ns = _feed.feed_reads_mt(fn, size_fn, flat, n_mhs, len(mh_groups), _vp(reads), n_reads, stride, force, warm_reads)
    _check()
    return ns * 1e-9


class Signature:
    """Signature (lib.rs:546-565) behind signature_* (ffi.rs:327-534)."""

    def __init__(self, _ptr=None):
        self._p = _ptr if _ptr is not None else _call("signature_new")

    def __del__(self):
        p, self._p = getattr(self, "_p", None), None
        if p and _lib is not None:
            _lib.signature_free(p)

    def set_name(self, name: str):
        _call("signature_set_name", self._p, name.encode())

    def set_filename(self, name: str):
        _call("signature_set_filename", self._p, name.encode())

    def push_mh(self, mh):
        _call("signature_push_mh", self._p, mh._p)

    def set_mh(self, mh):
        _call("signature_set_mh", self._p, mh._p)

    name = property(lambda s: _take_str(_call("signature_get_name", s._p)).decode())
    filename = property(lambda s: _take_str(_call("signature_get_filename", s._p)).decode())
    license = property(lambda s: _take_str(_call("signature_get_license", s._p)).decode())

    def first_mh(self):
        return KmerMinHash(0, 0, _ptr=_call("signature_first_mh", self._p))

    def mhs(self):
        n = usz(0)
        arr = _call("signature_get_mhs", self._p, C.byref(n))
        return [KmerMinHash(0, 0, _ptr=arr[i]) for i in range(n.value)]

    def __eq__(self, other):
        return bool(_call("signature_eq", self._p, other._p))

    __hash__ = None

    def save_json(self) -> bytes:
        return _take_str(_call("signature_save_json", self._p))


def signatures_save_buffer(sigs) -> bytes:
    arr = (vp * max(1, len(sigs)))(*[s._p for s in sigs])
    return _take_str(_call("signatures_save_buffer", arr, len(sigs)))


def _wrap_sigs(arr, n):
    return [Signature(_ptr=arr[i]) for i in range(n)]


def signatures_load_buffer(data: bytes, ksize=0, select_moltype=None, ignore_md5sum=False):
    n = usz(0)
    mt = None if select_moltype is None else select_moltype.encode()
    arr = _call("signatures_load_buffer", data, len(data), ignore_md5sum, ksize, mt, C.byref(n))
    return _wrap_sigs(arr, n.value)


def signatures_load_path(path: str, ksize=0, select_moltype=None, ignore_md5sum=False):
    n = usz(0)
    mt = None if select_moltype is None else select_moltype.encode()
    arr = _call("signatures_load_path", path.encode(), ignore_md5sum, ksize, mt, C.byref(n))
    return _wrap_sigs(arr, n.value)


class SketchCollection:
    """Packed CSR of sorted sketches in HBM (include/sourmash_b200.h)."""

    def __init__(self, _ptr=None):
        self._p = _ptr if _ptr is not None else _call("smgpu_collection_new")

    def __del__(self):
        p, self._p = getattr(self, "_p", None), None
        if p and _lib is not None:
            _lib.smgpu_collection_free(p)

    @classmethod
    def from_sketches(cls, mhs):
        c = cls()
        for m in mhs:
            c.push(m)
        return c

    @classmethod
    def from_csr(cls, hashes, offsets, n_rows, num, ksize, seed=42, max_hash=0, on_device=False):
        if not on_device:
            hashes = np.ascontiguousarray(hashes, dtype=np.uint64)
            offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        return cls(_ptr=_call("smgpu_collection_from_csr", _vp(hashes), _vp(offsets), n_rows, num, ksize, seed,
                              max_hash, on_device))

    @classmethod
    def sketch_sequences(cls, buf, offsets, num, ksize, seed=42, max_hash=0, on_device=False, n_seqs=None):
        """One fresh sketch per sequence buf[offsets[s]:offsets[s+1]], in one pass (smgpu_sketch_collection)."""
        if on_device:
            assert n_seqs is not None
            keep_b, keep_o = buf, offsets
        else:
            keep_b = buf if isinstance(buf, (int, np.ndarray)) else bytes(buf)
            keep_o = np.ascontiguousarray(offsets, dtype=np.uint64)
            n_seqs = keep_o.size - 1
        return cls(_ptr=_call("smgpu_sketch_collection", _vp(keep_b), _vp(keep_o), n_seqs, num, ksize, seed, max_hash, on_device))

    def rows_np(self):
        """The packed sketches as a list of numpy arrays (copies the CSR to the host)."""
        n = len(self)
        total = _call("smgpu_collection_copy", self._p, None, None)
        offs = np.zeros(n + 1, dtype=np.uint64)
        hashes = np.zeros(max(1, total), dtype=np.uint64)
        _call("smgpu_collection_copy", self._p, _vp(hashes), _vp(offs))
        return [hashes[int(offs[i]):int(offs[i + 1])].copy() for i in range(n)]

    def push(self, mh):
        _call("smgpu_collection_push", self._p, mh._p)

    @classmethod
    def from_signatures(cls, sigs):
        """One row per loaded signature (its first sketch), pushed in one call."""
        c = cls()
        arr = (vp * max(1, len(sigs)))(*[s._p for s in sigs])
        _call("smgpu_collection_push_signatures", c._p, arr, len(sigs))
        return c

    def __len__(self):
        return _call("smgpu_collection_len", self._p)

    def csr_device(self):
        h, o = vp(), vp()
        n = _call("smgpu_collection_csr", self._p, C.byref(h), C.byref(o))
        return h.value, o.value, n


def compare_matrix(rows, cols, mode="compare", r0=0, nr=None, c0=0, nc=None, want=("common", "size", "ratio")):
    """Block of the all-vs-all matrix as numpy arrays (host output)."""
    nr = len(rows) - r0 if nr is None else nr
    nc = len(cols) - c0 if nc is None else nc
    common = np.zeros((nr, nc), dtype=np.uint32) if "common" in want else None
    size = np.zeros((nr, nc), dtype=np.uint32) if "size" in want else None
    ratio = np.zeros((nr, nc), dtype=np.float64) if "ratio" in want else None
    _call("smgpu_compare_matrix", rows._p, r0, nr, cols._p, c0, nc, 1 if mode == "containment" else 0, _vp(common),
          _vp(size), _vp(ratio), nc, False)
    return common, size, ratio


def compare_matrix_device(rows, cols, mode, r0, nr, c0, nc, common_ptr, size_ptr, ratio_ptr, ld):
    """Same, writing into device memory the caller owns (raw pointers, e.g. torch tensors' data_ptr())."""
    _call("smgpu_compare_matrix", rows._p, r0, nr, cols._p, c0, nc, 1 if mode == "containment" else 0,
          _vp(common_ptr), _vp(size_ptr), _vp(ratio_ptr), ld, True)


def scaffold_pairs(coll):
    """Leaf-pairing pass of scaffold (sbt.rs:356-381): [(next_leaf, similar_leaf | None)] in processing order."""
    n = len(coll)
    a, b = np.zeros(max(1, (n + 1) // 2), dtype=np.uint64), np.zeros(max(1, (n + 1) // 2), dtype=np.uint64)
    k = _call("smgpu_scaffold_pairs", coll._p, _vp(a), _vp(b))
    return [(int(a[i]), None if b[i] == np.uint64(0xFFFFFFFFFFFFFFFF) else int(b[i])) for i in range(k)]


def linear_find(index, queries, mode, threshold, hits_cap=None):
    """LinearIndex::find for every query (linear.rs:25-45); returns a list of hit-id lists."""
    nq = len(queries)
    cap = hits_cap if hits_cap is not None else max(1, len(index) * nq)
    offs = np.zeros(nq + 1, dtype=np.uint64)
    hits = np.zeros(cap, dtype=np.uint64)
    total = _call("smgpu_linear_find", index._p, queries._p, 1 if mode == "containment" else 0, float(threshold),
                  _vp(offs), _vp(hits), cap)
    assert total <= cap
    return [hits[int(offs[q]):int(offs[q + 1])].tolist() for q in range(nq)]


# ---- multi-GPU (one process per GPU; NCCL inside the library) -------------------------------------------------
def comm_unique_id() -> bytes:
    buf = np.zeros(128, dtype=np.uint8)
    _call("smgpu_comm_unique_id", _vp(buf))
    return buf.tobytes()


def comm_init(id_bytes: bytes, rank: int, world: int):
    assert len(id_bytes) == 128
    _call("smgpu_comm_init", _vp(np.frombuffer(id_bytes, dtype=np.uint8).copy()), rank, world)


def comm_init_from_torch():
    """Convenience for hosts that already run torch.distributed: rank 0 makes the id, broadcast hands it round."""
    import torch
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    t = torch.zeros(128, dtype=torch.uint8)
    if rank == 0:
        t = torch.from_numpy(np.frombuffer(comm_unique_id(), dtype=np.uint8).copy())
    t = t.to(dev)
    dist.broadcast(t, 0)
    comm_init(t.cpu().numpy().tobytes(), rank, world)


def comm_destroy():
    _call("smgpu_comm_destroy")


def comm_rank_world():
    return lib().smgpu_comm_rank(), lib().smgpu_comm_world()


def collection_allgather(local):
    return SketchCollection(_ptr=_call("smgpu_collection_allgather", local._p))


def compare_matrix_allgather_device(local, mode, common_ptr, size_ptr, ratio_ptr, ld):
    """This rank's row block (local rows x all ranks' rows) into device memory; returns the gathered collection."""
    return SketchCollection(_ptr=_call("smgpu_compare_matrix_allgather", local._p, 1 if mode == "containment" else 0,
                                       _vp(common_ptr), _vp(size_ptr), _vp(ratio_ptr), ld, True))


def comm_allmerge(mh):
    _call("smgpu_comm_allmerge", mh._p)


def linear_find_sharded(index_part, queries, mode, threshold, hits_cap):
    nq = len(queries)
    offs = np.zeros(nq + 1, dtype=np.uint64)
    hits = np.zeros(max(1, hits_cap), dtype=np.uint64)
    total = _call("smgpu_linear_find_sharded", index_part._p, queries._p, 1 if mode == "containment" else 0, float(threshold),
                  _vp(offs), _vp(hits), hits_cap)
    assert total <= hits_cap
    return [hits[int(offs[q]):int(offs[q + 1])].tolist() for q in range(nq)]


class Nodegraph:
    """Nodegraph (src/index/nodegraph.rs:11-225) with its bitsets in HBM, behind smgpu_nodegraph_*."""

    def __init__(self, tablesizes=None, ksize=0, _ptr=None):
        if _ptr is not None:
            self._p = _ptr
        else:
            ts = np.ascontiguousarray(tablesizes, dtype=np.uint64)
            self._p = _call("smgpu_nodegraph_new", _vp(ts), ts.size, ksize)

    def __del__(self):
        p, self._p = getattr(self, "_p", None), None
        if p and _lib is not None:
            _lib.smgpu_nodegraph_free(p)

    @classmethod
    def from_buffer(cls, data: bytes):
        """Nodegraph::from_reader over a khmer OXLI v4 file image."""
        return cls(_ptr=_call("smgpu_nodegraph_from_buffer", data, len(data)))

    def save(self) -> bytes:
        n = _call("smgpu_nodegraph_save", self._p, None, 0)
        out = np.zeros(n, dtype=np.uint8)
        _call("smgpu_nodegraph_save", self._p, _vp(out), n)
        return out.tobytes()

    def count_many(self, hashes):
        """(number of new k-mers, per-hash return value of Nodegraph::count in batch order)"""
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        flags = np.zeros(h.size, dtype=np.uint8)
        n = _call("smgpu_nodegraph_count_many", self._p, _vp(h), h.size, _vp(flags), False) if h.size else 0
        return n, flags.astype(bool)

    def count(self, h):
        return bool(self.count_many([h])[1][0])

    def get_many(self, hashes):
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        flags = np.zeros(h.size, dtype=np.uint8)
        n = _call("smgpu_nodegraph_get_many", self._p, _vp(h), h.size, _vp(flags), False) if h.size else 0
        return n, flags

    def get(self, h):
        return int(self.get_many([h])[1][0])

    def matches(self, mh):
        return _call("smgpu_nodegraph_matches", self._p, mh._p)

    def update(self, other):
        _call("smgpu_nodegraph_update", self._p, other._p)

    def similarity(self, other):
        return _call("smgpu_nodegraph_similarity", self._p, other._p)

    def containment(self, other):
        return _call("smgpu_nodegraph_containment", self._p, other._p)

    def tablesizes(self):
        n = _call("smgpu_nodegraph_tablesizes", self._p, None, 0)
        out = np.zeros(max(1, n), dtype=np.uint64)
        _call("smgpu_nodegraph_tablesizes", self._p, _vp(out), n)
        return [int(x) for x in out[:n]]

    def ksize(self):
        return _call("smgpu_nodegraph_ksize", self._p)

    def n_occupied_bins(self):
        return _call("smgpu_nodegraph_n_occupied_bins", self._p)

    def unique_kmers(self):
        return _call("smgpu_nodegraph_unique_kmers", self._p)


def sbt_find(d, nodes, leaf_positions, leaves, queries, mode="similarity", threshold=0.0):
    """SBT::find (src/index/sbt.rs:147-175) for every row of `queries`.
    nodes: {position: (Nodegraph, min_n_below)}; leaves: SketchCollection whose row i sits at leaf_positions[i].
    Returns, per query, the positions of the matching leaves in the reference's visit order."""
    npos = sorted(nodes)
    a_np = np.ascontiguousarray(npos, dtype=np.uint64)
    a_ng = (C.c_void_p * max(1, len(npos)))(*[nodes[p][0]._p for p in npos])
    a_mb = np.ascontiguousarray([nodes[p][1] for p in npos], dtype=np.uint64)
    a_lp = np.ascontiguousarray(leaf_positions, dtype=np.uint64)
    nq = len(queries)
    offs = np.zeros(nq + 1, dtype=np.uint64)
    cap = max(1, nq * max(1, len(leaf_positions)))
    hits = np.zeros(cap, dtype=np.uint64)
    _call("smgpu_sbt_find", d, _vp(a_np), C.cast(a_ng, C.c_void_p), _vp(a_mb), len(npos), _vp(a_lp), leaves._p, queries._p,
          1 if mode == "containment" else 0, threshold, _vp(offs), _vp(hits), cap)
    return [[int(x) for x in hits[int(offs[q]):int(offs[q + 1])]] for q in range(nq)]
