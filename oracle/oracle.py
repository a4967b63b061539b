"""ctypes binding of the test-only CPU oracle (oracle/oracle.c, baseline_mt.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and
bench.py's cpu_baseline / --impl reference legs -- never by the product
package.  Mirrors the reference's crate API names (KmerMinHash::new,
add_sequence, add_hash, merge, compare, count_common, ...; src/lib.rs:141-513).
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "liboracle.so")


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("oracle.c", "baseline_mt.c", "Makefile")]
    stale = (not os.path.exists(_SO)) or any(os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE, "-B", "liboracle.so"], stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        u64, u32, sz, vp, i = C.c_uint64, C.c_uint32, C.c_size_t, C.c_void_p, C.c_int
        sig = {
            "orc_hash_murmur": (u64, [C.c_char_p, sz, u64]),
            "orc_smhasher_verification": (u32, []),
            "orc_mh_new": (vp, [u32, u32, i, u64, u64, i]),
            "orc_mh_free": (None, [vp]),
            "orc_mh_clone": (vp, [vp]),
            "orc_mh_size": (sz, [vp]),
            "orc_mh_mins": (C.POINTER(u64), [vp]),
            "orc_mh_abunds_size": (sz, [vp]),
            "orc_mh_abunds": (C.POINTER(u64), [vp]),
            "orc_mh_track_abundance": (i, [vp]),
            "orc_mh_mins_push": (None, [vp, u64]),
            "orc_mh_abunds_push": (None, [vp, u64]),
            "orc_mh_check_compatible": (i, [vp, vp]),
            "orc_mh_add_hash": (None, [vp, u64]),
            "orc_mh_add_word": (None, [vp, C.c_char_p, sz]),
            "orc_mh_add_sequence": (i, [vp, C.c_char_p, sz, i, C.c_char_p]),
            "orc_mh_add_many": (None, [vp, C.POINTER(u64), sz]),
            "orc_mh_add_from": (None, [vp, vp]),
            "orc_mh_add_reads": (i, [vp, C.c_char_p, sz, sz, i]),
            "orc_mh_merge": (i, [vp, vp]),
            "orc_mh_count_common": (i, [vp, vp, C.POINTER(u64)]),
            "orc_mh_intersection_size": (i, [vp, vp, C.POINTER(u64), C.POINTER(u64)]),
            "orc_mh_intersection": (i, [vp, vp, C.POINTER(u64), sz, C.POINTER(u64), C.POINTER(u64)]),
            "orc_mh_compare": (i, [vp, vp, C.POINTER(C.c_double)]),
            "orc_leaf_similarity": (C.c_double, [vp, vp]),
            "orc_leaf_containment": (C.c_double, [vp, vp]),
            "orc_linear_find": (sz, [C.POINTER(vp), sz, vp, i, C.c_double, C.POINTER(u64)]),
            "orc_compare_matrix": (None, [C.POINTER(vp), sz, C.POINTER(vp), sz, vp, vp, vp]),
            "orc_count_common_matrix": (None, [C.POINTER(vp), sz, C.POINTER(vp), sz, vp]),
            "orc_scaffold_pairs": (sz, [C.POINTER(vp), sz, C.POINTER(u64), C.POINTER(u64)]),
            "orc_md5_hex": (None, [C.c_char_p, sz, C.c_char_p]),
            "orc_mh_md5sum": (None, [vp, C.c_char_p]),
            "orc_signature_json": (vp, [C.c_char_p, C.c_char_p, C.POINTER(vp), sz]),
            "orc_free": (None, [vp]),
            "orc_mt_sketch_reads": (None, [C.c_char_p, sz, sz, C.POINTER(u32), i, u32, u64, i, i, C.POINTER(vp)]),
            "orc_mt_sketch_each": (None, [C.c_char_p, vp, sz, u32, u32, i, u64, u64, i, i, C.POINTER(vp)]),
            "orc_mt_compare_matrix": (None, [C.POINTER(vp), sz, C.POINTER(vp), sz, vp, vp, i]),
            "orc_mt_compare_pairs": (None, [C.POINTER(vp), vp, vp, sz, vp, vp, i]),
            "orc_ng_new": (vp, [C.POINTER(u64), sz, sz]),
            "orc_ng_free": (None, [vp]),
            "orc_ng_count": (i, [vp, u64]),
            "orc_ng_get": (sz, [vp, u64]),
            "orc_ng_count_many": (u64, [vp, vp, sz, vp]),
            "orc_ng_get_many": (u64, [vp, vp, sz, vp]),
            "orc_ng_update": (i, [vp, vp]),
            "orc_ng_save": (sz, [vp, C.c_char_p, sz]),
            "orc_ng_load": (vp, [C.c_char_p, sz]),
            "orc_ng_n_tables": (sz, [vp]),
            "orc_ng_tablesize": (u64, [vp, sz]),
            "orc_ng_ksize": (sz, [vp]),
            "orc_ng_occupied_bins": (sz, [vp]),
            "orc_ng_unique_kmers": (sz, [vp]),
            "orc_ng_blocks": (C.POINTER(u32), [vp, sz]),
            "orc_ng_similarity": (C.c_double, [vp, vp]),
            "orc_ng_containment": (C.c_double, [vp, vp]),
            "orc_ng_matches": (u64, [vp, vp]),
            "orc_node_similarity": (C.c_double, [vp, u64, vp]),
            "orc_node_containment": (C.c_double, [vp, vp]),
            "orc_sbt_new": (vp, [u32, vp, vp, vp, sz, vp, vp, sz]),
            "orc_sbt_free": (None, [vp]),
            "orc_sbt_query": (sz, [vp, vp, i, C.c_double, vp]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


class SourmashError(Exception):
    def __init__(self, code, message=""):
        super().__init__(f"[{code}] {message}")
        self.code = code
        self.message = message


_MESSAGES = {  # src/errors.rs:6-25
    101: "different ksizes cannot be compared",
    102: "DNA/prot minhashes cannot be compared",
    103: "mismatch in max_hash; comparison fail",
    104: "mismatch in seed; comparison fail",
}


def hash_murmur(kmer: bytes, seed: int = 42) -> int:
    return lib().orc_hash_murmur(kmer, len(kmer), seed)


class KmerMinHash:
    """Oracle sketch; same constructor order as KmerMinHash::new (lib.rs:142-149)."""

    def __init__(self, num, ksize, is_protein=False, seed=42, max_hash=0, track_abundance=False, _ptr=None):
        self._L = lib()
        self._p = _ptr if _ptr is not None else self._L.orc_mh_new(
            num, ksize, int(is_protein), seed, max_hash, int(track_abundance))
        self.num, self.ksize, self.is_protein, self.seed, self.max_hash = num, ksize, is_protein, seed, max_hash

    def __del__(self):
        if getattr(self, "_p", None):
            self._L.orc_mh_free(self._p)
            self._p = None

    def clone(self):
        return KmerMinHash(self.num, self.ksize, self.is_protein, self.seed, self.max_hash,
                           _ptr=self._L.orc_mh_clone(self._p))

    @property
    def mins(self):
        n = self._L.orc_mh_size(self._p)
        p = self._L.orc_mh_mins(self._p)
        return [p[i] for i in range(n)]

    @property
    def abunds(self):
        if not self._L.orc_mh_track_abundance(self._p):
            return None
        n = self._L.orc_mh_abunds_size(self._p)
        p = self._L.orc_mh_abunds(self._p)
        return [p[i] for i in range(n)]

    def mins_np(self):
        import numpy as np
        n = self._L.orc_mh_size(self._p)
        if n == 0:
            return np.zeros(0, dtype=np.uint64)
        return np.ctypeslib.as_array(self._L.orc_mh_mins(self._p), shape=(n,)).copy()

    def abunds_np(self):
        import numpy as np
        if not self._L.orc_mh_track_abundance(self._p):
            return None
        n = self._L.orc_mh_abunds_size(self._p)
        if n == 0:
            return np.zeros(0, dtype=np.uint64)
        return np.ctypeslib.as_array(self._L.orc_mh_abunds(self._p), shape=(n,)).copy()

    def size(self):
        return self._L.orc_mh_size(self._p)

    def track_abundance(self):
        return bool(self._L.orc_mh_track_abundance(self._p))

    def add_hash(self, h):
        self._L.orc_mh_add_hash(self._p, h)

    def add_many(self, hashes):
        import numpy as np
        a = np.ascontiguousarray(hashes, dtype=np.uint64)
        self._L.orc_mh_add_many(self._p, a.ctypes.data_as(C.POINTER(C.c_uint64)), a.size)

    def add_word(self, w: bytes):
        self._L.orc_mh_add_word(self._p, w, len(w))

    def add_sequence(self, seq: bytes, force=False):
        bad = C.create_string_buffer(self.ksize + 1)
        e = self._L.orc_mh_add_sequence(self._p, seq, len(seq), int(force), bad)
        if e == 1101:
            raise SourmashError(e, "invalid DNA character in input k-mer: " + bad.value.decode("latin-1"))
        if e:
            raise SourmashError(e, "unsupported")

    def add_reads(self, buf: bytes, nreads, readlen, force=True):
        e = self._L.orc_mh_add_reads(self._p, buf, nreads, readlen, int(force))
        if e:
            raise SourmashError(e)

    def add_from(self, other):
        self._L.orc_mh_add_from(self._p, other._p)

    def mins_push(self, v):
        self._L.orc_mh_mins_push(self._p, v)

    def abunds_push(self, v):
        self._L.orc_mh_abunds_push(self._p, v)

    def merge(self, other):
        e = self._L.orc_mh_merge(self._p, other._p)
        if e:
            raise SourmashError(e, _MESSAGES.get(e, ""))

    def count_common(self, other):
        c = C.c_uint64()
        e = self._L.orc_mh_count_common(self._p, other._p, C.byref(c))
        if e:
            raise SourmashError(e, _MESSAGES.get(e, ""))
        return c.value

    def intersection_size(self, other):
        c, s = C.c_uint64(), C.c_uint64()
        e = self._L.orc_mh_intersection_size(self._p, other._p, C.byref(c), C.byref(s))
        if e:
            raise SourmashError(e, _MESSAGES.get(e, ""))
        return c.value, s.value

    def intersection(self, other):  # lib.rs:438-468
        cap = min(self.size(), other.size())
        buf = (C.c_uint64 * max(1, cap))()
        n, s = C.c_uint64(), C.c_uint64()
        e = self._L.orc_mh_intersection(self._p, other._p, buf, cap, C.byref(n), C.byref(s))
        if e:
            raise SourmashError(e, _MESSAGES.get(e, ""))
        return np.array(buf[:n.value], dtype=np.uint64), s.value

    def compare(self, other):
        d = C.c_double()
        e = self._L.orc_mh_compare(self._p, other._p, C.byref(d))
        if e:
            raise SourmashError(e, _MESSAGES.get(e, ""))
        return d.value

    def similarity(self, other):  # Leaf<Signature>::similarity, index.rs:131-144
        return self._L.orc_leaf_similarity(self._p, other._p)

    def containment(self, other):  # Leaf<Signature>::containment, index.rs:146-160
        return self._L.orc_leaf_containment(self._p, other._p)

    def md5sum(self):
        out = C.create_string_buffer(33)
        self._L.orc_mh_md5sum(self._p, out)
        return out.value.decode()


def _ptr_array(mhs):
    arr = (C.c_void_p * len(mhs))(*[m._p for m in mhs])
    return arr


def linear_find(leaves, query, mode, threshold):
    """LinearIndex::find (linear.rs:25-45); mode 'similarity' | 'containment' (search.rs:3-9)."""
    hits = (C.c_uint64 * max(1, len(leaves)))()
    n = lib().orc_linear_find(_ptr_array(leaves), len(leaves), query._p,
                              1 if mode == "containment" else 0, threshold, hits)
    return [hits[i] for i in range(n)]


def scaffold_pairs(leaves):
    """Leaf-pairing pass of scaffold (sbt.rs:356-381): [(next_leaf, similar_leaf | None)] in processing order."""
    n = len(leaves)
    a, b = (C.c_uint64 * max(1, n))(), (C.c_uint64 * max(1, n))()
    k = lib().orc_scaffold_pairs(_ptr_array(leaves), n, a, b)
    return [(a[i], None if b[i] == 0xFFFFFFFFFFFFFFFF else b[i]) for i in range(k)]


def sketch_each(buf: bytes, offsets, num, ksize, is_protein=False, seed=42, max_hash=0, track_abundance=False,
                nthreads=None):
    """One fresh sketch per sequence buf[offsets[s]:offsets[s+1]] (new + add_sequence(force=True)), the sequences
    spread over nthreads host threads (default: every CPU); returns [KmerMinHash] in sequence order."""
    o = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = o.size - 1
    assert n >= 0 and (n == 0 or int(o[-1]) <= len(buf))
    out = (C.c_void_p * max(1, n))()
    lib().orc_mt_sketch_each(buf, o.ctypes.data, n, num, ksize, int(is_protein), seed, max_hash, int(track_abundance),
                             nthreads or os.cpu_count() or 4, out)
    return [KmerMinHash(num, ksize, is_protein, seed, max_hash, track_abundance, _ptr=out[s]) for s in range(n)]


def compare_matrix(rows, cols, nthreads=1):
    import numpy as np
    common = np.zeros((len(rows), len(cols)), dtype=np.uint32)
    size = np.zeros((len(rows), len(cols)), dtype=np.uint32)
    lib().orc_mt_compare_matrix(_ptr_array(rows), len(rows), _ptr_array(cols), len(cols),
                                common.ctypes.data, size.ctypes.data, nthreads)
    return common, size


def compare_pairs(mhs, ia, ib, nthreads=1):
    """(common, size) of KmerMinHash::compare for the pairs (mhs[ia[p]], mhs[ib[p]])"""
    ia = np.ascontiguousarray(ia, dtype=np.uint64)
    ib = np.ascontiguousarray(ib, dtype=np.uint64)
    common = np.zeros(len(ia), dtype=np.uint32)
    size = np.zeros(len(ia), dtype=np.uint32)
    lib().orc_mt_compare_pairs(_ptr_array(mhs), ia.ctypes.data, ib.ctypes.data, len(ia), common.ctypes.data, size.ctypes.data,
                               nthreads)
    return common, size


def count_common_matrix(rows, cols):
    import numpy as np
    common = np.zeros((len(rows), len(cols)), dtype=np.uint32)
    lib().orc_count_common_matrix(_ptr_array(rows), len(rows), _ptr_array(cols), len(cols), common.ctypes.data)
    return common


def signature_json(mhs, name=None, filename=None) -> bytes:
    L = lib()
    p = L.orc_signature_json(None if name is None else name.encode(), None if filename is None else filename.encode(),
                             _ptr_array(mhs), len(mhs))
    s = C.string_at(p)
    L.orc_free(p)
    return s


def md5_hex(data: bytes) -> str:
    out = C.create_string_buffer(33)
    lib().orc_md5_hex(data, len(data), out)
    return out.value.decode()


def mt_sketch_reads(buf: bytes, nreads, readlen, ksizes, num, max_hash, track_abundance, nthreads):
    """CPU baseline: sketch fixed-length reads on nthreads host threads; returns [KmerMinHash] per ksize."""
    L = lib()
    ks = (C.c_uint32 * len(ksizes))(*ksizes)
    out = (C.c_void_p * len(ksizes))()
    L.orc_mt_sketch_reads(buf, nreads, readlen, ks, len(ksizes), num, max_hash, int(track_abundance), nthreads, out)
    return [KmerMinHash(num, k, False, 42, max_hash, track_abundance, _ptr=out[i]) for i, k in enumerate(ksizes)]


class Nodegraph:
    """Oracle khmer bloom filter (src/index/nodegraph.rs:11-225)."""

    def __init__(self, tablesizes=None, ksize=0, _ptr=None):
        self._L = lib()
        if _ptr is not None:
            self._p = _ptr
        else:
            ts = (C.c_uint64 * max(1, len(tablesizes)))(*tablesizes)
            self._p = self._L.orc_ng_new(ts, len(tablesizes), ksize)

    def __del__(self):
        if getattr(self, "_p", None):
            self._L.orc_ng_free(self._p)
            self._p = None

    @classmethod
    def from_buffer(cls, data: bytes):
        p = lib().orc_ng_load(data, len(data))
        if not p:
            raise SourmashError(1, "Nodegraph::from_reader failed")
        return cls(_ptr=p)

    def save(self) -> bytes:
        n = self._L.orc_ng_save(self._p, None, 0)
        buf = C.create_string_buffer(n)
        self._L.orc_ng_save(self._p, buf, n)
        return buf.raw

    def count(self, h):
        return bool(self._L.orc_ng_count(self._p, h))

    def get(self, h):
        return self._L.orc_ng_get(self._p, h)

    def count_many(self, hashes):
        """(number of new k-mers, count(h) for each hash in batch order as a bool array)"""
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        flags = np.zeros(h.size, dtype=np.uint8)
        n = self._L.orc_ng_count_many(self._p, h.ctypes.data, h.size, flags.ctypes.data)
        return n, flags.astype(bool)

    def get_many(self, hashes):
        """(sum of get(h), get(h) for each hash as a uint8 array)"""
        h = np.ascontiguousarray(hashes, dtype=np.uint64)
        flags = np.zeros(h.size, dtype=np.uint8)
        n = self._L.orc_ng_get_many(self._p, h.ctypes.data, h.size, flags.ctypes.data)
        return n, flags

    def update(self, other):
        if self._L.orc_ng_update(self._p, other._p):
            raise SourmashError(1, "FixedBitSet::put out of bounds")

    def tablesizes(self):
        return [self._L.orc_ng_tablesize(self._p, t) for t in range(self._L.orc_ng_n_tables(self._p))]

    def ksize(self):
        return self._L.orc_ng_ksize(self._p)

    def n_occupied_bins(self):
        return self._L.orc_ng_occupied_bins(self._p)

    def unique_kmers(self):
        return self._L.orc_ng_unique_kmers(self._p)

    def bit(self, t, i):
        """bit i of table t"""
        return (self._L.orc_ng_blocks(self._p, t)[i >> 5] >> (i & 31)) & 1

    def similarity(self, other):
        return self._L.orc_ng_similarity(self._p, other._p)

    def containment(self, other):
        return self._L.orc_ng_containment(self._p, other._p)

    def matches(self, mh):
        return self._L.orc_ng_matches(self._p, mh._p)


def node_similarity(ng, min_n_below, query):  # sbt.rs:233-254
    return lib().orc_node_similarity(ng._p, min_n_below, query._p)


def node_containment(ng, query):  # sbt.rs:256-277
    return lib().orc_node_containment(ng._p, query._p)


class SbtOracle:
    """An SBT indexed once for many SBT::find walks (sbt.rs:147-175).  The tree is given by position as lists, so
    that a position may be listed twice (its first entry wins): node_positions[i] holds Nodegraph nodes[i] with
    min_n_below[i], leaf_positions[i] holds KmerMinHash leaves[i]."""

    def __init__(self, d, node_positions, nodes, min_n_below, leaf_positions, leaves):
        self._L = lib()
        self._keep = (list(nodes), list(leaves))  # the C index borrows them
        self.n_leaves = len(leaves)
        npos = np.ascontiguousarray(node_positions, dtype=np.uint64)
        mnb = np.ascontiguousarray(min_n_below, dtype=np.uint64)
        lpos = np.ascontiguousarray(leaf_positions, dtype=np.uint64)
        assert npos.size == mnb.size == len(nodes) and lpos.size == len(leaves)
        self._p = self._L.orc_sbt_new(d, npos.ctypes.data, C.cast(_ptr_array(nodes), C.c_void_p), mnb.ctypes.data, npos.size,
                                      lpos.ctypes.data, C.cast(_ptr_array(leaves), C.c_void_p), lpos.size)

    def __del__(self):
        if getattr(self, "_p", None):
            self._L.orc_sbt_free(self._p)
            self._p = None

    def find(self, query, mode, threshold):
        """positions of the matching leaves in visit order; mode 'similarity' | 'containment'"""
        hits = np.zeros(max(1, self.n_leaves), dtype=np.uint64)
        n = self._L.orc_sbt_query(self._p, query._p, 1 if mode == "containment" else 0, threshold, hits.ctypes.data)
        return [int(x) for x in hits[:n]]


def sbt_find(d, nodes, leaves, query, mode, threshold):
    """SBT::find (sbt.rs:147-175).  nodes: {position: (Nodegraph, min_n_below)}, leaves: {position: KmerMinHash};
    returns the positions of the matching leaves in visit order."""
    npos, lpos = sorted(nodes), sorted(leaves)
    tree = SbtOracle(d, npos, [nodes[p][0] for p in npos], [nodes[p][1] for p in npos], lpos, [leaves[p] for p in lpos])
    return tree.find(query, mode, threshold)
