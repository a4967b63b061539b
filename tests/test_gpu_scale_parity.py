"""GPU parity at the shapes where the host code changes plan, and at the hash values it special-cases.

The other GPU tests check the C ABI bit for bit against the oracle at small shapes, inside one block of every
blocked loop.  Here the collections are large enough to cross each threshold of csrc/collection.cu (the pair list
sized from a host read, the double-buffered host output, linear_find's index blocks, the automatic choice of the
index-streaming search), and every test asserts the shape fact that puts it past its threshold, so that a change of
a constant shows up as a failure instead of a test that quietly stops reaching its branch.

The all-vs-all references are exact and whole-matrix without an O(N^2) oracle walk: the collections are planted
clusters with disjoint hash pools, so every cross-cluster cell is unrelated by construction and only the clusters
go through the oracle (oracle/oracle.c).  Search references come from a sparse incidence product.
"""
import contextlib
import os

import numpy as np
import pytest
import scipy.sparse as sp

import sourmash_rust_b200 as smb
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

# csrc/collection.cu
PAIR_LIST_DEVICE_CELLS = 1 << 26    # compare_block_device: a larger block sizes its related-pair list from a host read
HOST_BLOCK_CELLS = 1 << 25          # compare_matrix, host outputs: row blocks of at most this many cells
FIND_BLOCK_CELLS = 1 << 27          # linear_find: index blocks of FIND_BLOCK_CELLS / nq rows
STREAM_MIN_INDEX_HASHES = 1 << 22   # linear_find 'auto' streams an index of at least this many hashes ...
STREAM_INDEX_OVER_QUERY = 4         # ... holding at least this many times the query hashes
# csrc/find_stream.cu
STREAM_MULTI_SLICE_AVG_LEN = 200    # find_stream_partitions: more than one slice from rows of 200 hashes on average
QT_SLICES = 1024                    # table slices of the query hashes
QT_SMEM_SLOTS = 12288               # a table slice of more slots (2 per posting + 32) is built in place in global memory
# csrc/sortops.cu
FOLD_SMALL = 2048                   # at most this many new hashes fold through fold_small_sort_kernel

U64_MAX = (1 << 64) - 1
SCALED_MAX_HASH = 1 << 63
EDGE = np.array([0, 1, 2**32 - 1, 2**32, 2**63 - 1, 2**63, 2**64 - 2, 2**64 - 1], dtype=np.uint64)
NTHREADS = max(1, min(16, os.cpu_count() or 1))
U32_SENTINEL = 0xA5A5A5A5
F64_SENTINEL = -7.25


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


@contextlib.contextmanager
def knobs(compare=None, find=None):
    """Sets the library's path knobs for the block and always puts them back."""
    try:
        if compare:
            smb.compare_path(compare)
        if find:
            smb.find_path(find)
        yield
    finally:
        if compare:
            smb.compare_path("auto")
        if find:
            smb.find_path("auto")


def mismatch(name, got, want):
    """'' when equal (NaN equals NaN), else how many cells differ and where the first ones are."""
    assert got.shape == want.shape, (name, got.shape, want.shape)
    if got.dtype.kind == "f":
        bad = ~((got == want) | (np.isnan(got) & np.isnan(want)))
    else:
        bad = got != want
    n = int(np.count_nonzero(bad))
    if not n:
        return ""
    at = np.argwhere(bad)[:5]
    return f"{name}: {n} cells differ, first at {at.tolist()}: got {got[tuple(at.T)].tolist()} want {want[tuple(at.T)].tolist()}"


# ------------------------------------------------------------------------------------------------
# planted collections
# ------------------------------------------------------------------------------------------------
class Planted:
    """Clusters of 30-150 sketches, each cluster drawing from a hash pool of its own; rows shuffled.

    values: every pool hash (pool id -> hash), ids[k]: the pool ids of row k (ascending hash), cid[k]: its cluster."""

    def __init__(self, n_rows, num, max_hash, seed, *, full_len=0, len_range=(20, 3000), log_len=True, pool=3300,
                 n_empty=0, n_single=0, extra_pool=0):
        rng = np.random.Generator(np.random.PCG64(seed))
        sizes = []
        while sum(sizes) < n_rows:
            sizes.append(int(rng.integers(30, 151)))
        sizes[-1] -= sum(sizes) - n_rows
        pools = [int(rng.integers(full_len + 20, 3 * full_len)) if full_len else pool for _ in sizes]
        pstart = np.concatenate([[0], np.cumsum(pools)]).astype(np.int64)
        n_pool = int(pstart[-1])
        hi = (max_hash - 1) if max_hash else U64_MAX
        self.values = rng.integers(0, hi, size=n_pool + extra_pool, dtype=np.uint64, endpoint=True)
        # every pool hash is distinct: no hash occurs in two clusters (a collision means: pick another seed)
        assert np.unique(self.values).size == self.values.size
        self.extra = np.arange(n_pool, n_pool + extra_pool, dtype=np.int64)   # hashes of no cluster
        self.cluster_ids = []                                                 # per cluster: pool ids by ascending hash
        rows = []
        for c, m in enumerate(sizes):
            p0, pc = int(pstart[c]), pools[c]
            by_value = p0 + np.argsort(self.values[p0:p0 + pc], kind="stable")
            self.cluster_ids.append(by_value)
            if full_len:
                pick = np.sort(np.argpartition(rng.random((m, pc)), full_len - 1, axis=1)[:, :full_len], axis=1)
                rows.extend(by_value[pick])
            else:
                lo, hi_len = len_range
                want = np.exp(rng.uniform(np.log(lo), np.log(hi_len), m)) if log_len else rng.uniform(lo, hi_len, m)
                mask = rng.random((m, pc)) < (want / pc)[:, None]
                rows.extend(by_value[np.flatnonzero(r)] for r in mask)
        special = rng.choice(n_rows, n_empty + n_single, replace=False)
        for k in special[:n_empty]:
            rows[k] = rows[k][:0]
        for k in special[n_empty:]:
            rows[k] = rows[k][:1]
        perm = rng.permutation(n_rows)
        self.ids = [rows[k] for k in perm]
        self.cid = np.repeat(np.arange(len(sizes)), sizes)[perm]
        self.n, self.num, self.max_hash, self.n_clusters = n_rows, num, max_hash, len(sizes)
        self.lens = np.array([len(r) for r in self.ids], dtype=np.uint32)
        self.offsets = np.concatenate([[0], np.cumsum(self.lens, dtype=np.uint64)]).astype(np.uint64)
        self.hashes = self.values[np.concatenate(self.ids)] if n_rows else np.zeros(0, np.uint64)
        self.n_hashes = int(self.offsets[-1])
        self._coll = None

    def collection(self, ksize=31):
        if ksize != 31:
            return smb.SketchCollection.from_csr(self.hashes, self.offsets, self.n, self.num, ksize, 42, self.max_hash)
        if self._coll is None:
            self._coll = smb.SketchCollection.from_csr(self.hashes, self.offsets, self.n, self.num, 31, 42, self.max_hash)
        return self._coll

    def row(self, k):
        return self.hashes[int(self.offsets[k]):int(self.offsets[k + 1])]

    def oracle_sketch(self, k):
        o = orc.KmerMinHash(self.num, 31, False, 42, self.max_hash)
        o.add_many(self.row(k))
        assert o.size() == self.lens[k]
        return o

    def incidence(self, n_cols):
        """rows x pool ids, int64 ones"""
        cols = np.concatenate(self.ids).astype(np.int64) if self.n_hashes else np.zeros(0, np.int64)
        return sp.csr_matrix((np.ones(cols.size, np.int64), cols, self.offsets.astype(np.int64)), shape=(self.n, n_cols))


class Queries:
    """Query sketches given as pool ids of a Planted index (so that the incidence product is the count matrix)."""

    def __init__(self, base, ids, num=0):
        self.ids = ids
        self.n = len(ids)
        self.num, self.max_hash = num, base.max_hash
        self.lens = np.array([len(r) for r in ids], dtype=np.uint32)
        self.offsets = np.concatenate([[0], np.cumsum(self.lens, dtype=np.uint64)]).astype(np.uint64)
        self.hashes = base.values[np.concatenate(ids)]
        self.n_hashes = int(self.offsets[-1])
        self.n_pool = base.values.size

    def collection(self, ksize=31):
        return smb.SketchCollection.from_csr(self.hashes, self.offsets, self.n, self.num, ksize, 42, self.max_hash)

    def incidence(self):
        cols = np.concatenate(self.ids).astype(np.int64)
        return sp.csr_matrix((np.ones(cols.size, np.int64), cols, self.offsets.astype(np.int64)), shape=(self.n, self.n_pool))


def related_queries(base, nq, seed, num=0, fresh=20):
    """Each query: a random share of one cluster's pool and some hashes of no cluster, or (one in 16) a copy of an index
    sketch; a few duplicates, an empty query and a one-hash query."""
    rng = np.random.Generator(np.random.PCG64(seed))
    ids = []
    for q in range(nq):
        if q % 16 == 15:
            ids.append(base.ids[int(rng.integers(0, base.n))])
            continue
        pool = base.cluster_ids[int(rng.integers(0, base.n_clusters))]
        take = pool[rng.random(pool.size) < rng.uniform(0.05, 0.6)]
        extra = base.extra[rng.integers(0, base.extra.size, int(rng.integers(0, fresh + 1)))] if base.extra.size else take[:0]
        r = np.unique(np.concatenate([take, extra]))
        r = r[np.argsort(base.values[r], kind="stable")]
        if num:
            r = r[:num]
        ids.append(r)
    ids[3] = ids[3][:0]
    ids[4] = ids[4][:1]
    ids[5] = ids[2]
    ids[nq - 1] = ids[7]
    return ids


# ------------------------------------------------------------------------------------------------
# exact all-vs-all reference
# ------------------------------------------------------------------------------------------------
N_SQUARE = 8300
KINDS = ("full", "ragged")
MODES = ("compare", "containment")
_datasets = {}
_expected = {}


def square(kind):
    if kind not in _datasets:
        if kind == "full":   # every row holds exactly num = 500 hashes: the rank-compressed dense kernel applies
            ds = Planted(N_SQUARE, 500, 0, 0x5CA1E001, full_len=500)
        else:                # scaled sketches of 20-3000 hashes, a few empty and one-hash rows
            ds = Planted(N_SQUARE, 0, SCALED_MAX_HASH, 0x5CA1E002, n_empty=5, n_single=5)
        ds.clusters = []
        for c in range(ds.n_clusters):
            pos = np.flatnonzero(ds.cid == c)
            osk = [ds.oracle_sketch(k) for k in pos]
            oc, osz = orc.compare_matrix(osk, osk, NTHREADS)
            ds.clusters.append((pos, oc, osz, orc.count_common_matrix(osk, osk)))
        _datasets[kind] = ds
    return _datasets[kind]


def expected(kind, mode):
    """(common, size, ratio) of the whole N x N matrix; the last two (kind, mode) are kept (1.1 GB each)."""
    key = (kind, mode)
    if key not in _expected:
        while len(_expected) >= 2:
            del _expected[next(iter(_expected))]
        ds = square(kind)
        la = ds.lens
        common = np.zeros((ds.n, ds.n), dtype=np.uint32)
        if mode == "compare":
            # unrelated: common 0, size min(num, |A| + |B|) (|A| + |B| without a num)  (lib.rs:391-401)
            size = la[:, None] + la[None, :]
            if ds.num:
                np.minimum(size, np.uint32(ds.num), out=size)
        else:
            # unrelated: common 0, size |A| (the row sketch is the denominator, index.rs:152-154)
            size = np.repeat(la[:, None], ds.n, axis=1)
        for pos, oc, osz, occ in ds.clusters:
            ix = np.ix_(pos, pos)
            if mode == "compare":
                common[ix] = oc
                size[ix] = osz
            else:
                common[ix] = occ
        ratio = common.astype(np.float64)
        with np.errstate(invalid="ignore", divide="ignore"):
            np.true_divide(ratio, np.maximum(size, np.uint32(1)) if mode == "compare" else size, out=ratio)
        _expected[key] = (common, size, ratio)
    return _expected[key]


def check_block(got, want, rows=slice(None), cols=slice(None), what=""):
    msgs = []
    for name, g, w in zip(("common", "size", "ratio"), got, want):
        if g is not None:
            msgs.append(mismatch(f"{what} {name}", g, w[rows, cols]))
    msgs = [m for m in msgs if m]
    assert not msgs, "\n".join(msgs)


def padded(n_rows, ld, nc, dtype, sentinel):
    return np.full((n_rows, ld), sentinel, dtype=dtype)


def check_padding(buf, nc, sentinel, what):
    pad = buf[:, nc:]
    assert np.array_equal(pad, np.full_like(pad, sentinel)), f"{what}: padding columns overwritten"


# ------------------------------------------------------------------------------------------------
# (a) device outputs above 2^26 cells: host-sized pair list, symmetric walk through ld > nc
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("path", ["auto", "sparse", "dense"])
@pytest.mark.parametrize("kind", KINDS)
def test_device_outputs_whole_square(kind, path, mode):
    import torch
    ds = square(kind)
    N = ds.n
    assert N * N > PAIR_LIST_DEVICE_CELLS   # the sparse path sizes its pair list from the scan tail read on the host
    coll = ds.collection()
    want = expected(kind, mode)
    ld = N + 37

    def run(r0, nr):
        c = torch.full((nr, ld), U32_SENTINEL - (1 << 32), dtype=torch.int32, device="cuda")
        s = torch.full((nr, ld), U32_SENTINEL - (1 << 32), dtype=torch.int32, device="cuda")
        r = torch.full((nr, ld), F64_SENTINEL, dtype=torch.float64, device="cuda")
        torch.cuda.synchronize()
        with knobs(compare=path):
            smb.compare_matrix_device(coll, coll, mode, r0, nr, 0, N, c.data_ptr(), s.data_ptr(), r.data_ptr(), ld)
        out = [c.cpu().numpy().view(np.uint32), s.cpu().numpy().view(np.uint32), r.cpu().numpy()]
        del c, s, r
        for buf, sen, name in zip(out, (U32_SENTINEL, U32_SENTINEL, F64_SENTINEL), ("common", "size", "ratio")):
            check_padding(buf, N, sen, f"{kind}/{path}/{mode} r0={r0} {name}")
        check_block([o[:, :N] for o in out], want, slice(r0, r0 + nr), slice(None), f"{kind}/{path}/{mode} r0={r0}")

    run(0, N)          # the whole square: each unordered pair walked once, written to both cells
    run(1234, 3000)    # a rank's row shard against every column


# ------------------------------------------------------------------------------------------------
# (b) host outputs over three or more 2^25-cell row blocks: double buffering, strided copies, output subsets
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("path", ["auto", "sparse", "dense"])
@pytest.mark.parametrize("kind", KINDS)
def test_host_outputs_row_blocks(kind, path, mode):
    ds = square(kind)
    N = ds.n
    block_rows = HOST_BLOCK_CELLS // N
    assert -(-N // block_rows) >= 3   # three or more row blocks: the third waits on the first block's copy
    coll = ds.collection()
    want = expected(kind, mode)
    mode_i = 1 if mode == "containment" else 0
    with knobs(compare=path):
        got = smb.compare_matrix(coll, coll, mode)
        check_block(got, want, what=f"{kind}/{path}/{mode} contiguous")
        del got
        # one output at a time into a strided host matrix (ld > nc: the 2D copy); the others are null
        ld = N + 37
        for k, (name, dtype, sen) in enumerate((("common", np.uint32, U32_SENTINEL), ("size", np.uint32, U32_SENTINEL),
                                                ("ratio", np.float64, F64_SENTINEL))):
            buf = padded(N, ld, N, dtype, sen)
            ptrs = [None, None, None]
            ptrs[k] = buf
            smb._call("smgpu_compare_matrix", coll._p, 0, N, coll._p, 0, N, mode_i, smb._vp(ptrs[0]), smb._vp(ptrs[1]),
                      smb._vp(ptrs[2]), ld, False)
            check_padding(buf, N, sen, f"{kind}/{path}/{mode} {name} only")
            msg = mismatch(f"{kind}/{path}/{mode} {name} only", buf[:, :N], want[k])
            assert not msg, msg
            del buf
        # a rectangular block of two different collections: rows of this one against a shuffled subset of it
        rng = np.random.Generator(np.random.PCG64(7))
        sel = rng.choice(N, 5000, replace=False)
        other = smb.SketchCollection.from_csr(np.concatenate([ds.row(k) for k in sel]),
                                              np.concatenate([[0], np.cumsum(ds.lens[sel], dtype=np.uint64)]).astype(np.uint64),
                                              sel.size, ds.num, 31, 42, ds.max_hash)
        r0, nr = 100, 8000
        assert nr * sel.size > HOST_BLOCK_CELLS
        got = smb.compare_matrix(coll, other, mode, r0=r0, nr=nr)
    check_block(got, [w[:, sel] for w in want], slice(r0, r0 + nr), slice(None), f"{kind}/{path}/{mode} two collections")


# ------------------------------------------------------------------------------------------------
# linear_find references
# ------------------------------------------------------------------------------------------------
def find_raw(index, queries, mode, thr, cap):
    nq = len(queries)
    offs = np.zeros(nq + 1, dtype=np.uint64)
    hits = np.zeros(max(1, cap), dtype=np.uint64)
    total = smb._call("smgpu_linear_find", index._p, queries._p, 1 if mode == "containment" else 0, float(thr),
                      smb._vp(offs), smb._vp(hits), cap)
    assert total == offs[-1]
    return offs, hits[:min(total, cap)], total


def count_coo(index, queries):
    """|query n index row| of every pair sharing a hash: (q, i, count)"""
    m = (queries.incidence() @ index.incidence(queries.n_pool).T).tocoo()
    return m.row.astype(np.int64), m.col.astype(np.int64), m.data.astype(np.int64)


def hits_from_cells(nq, q, i, keep):
    q, i = q[keep], i[keep]
    order = np.lexsort((i, q))
    offs = np.concatenate([[0], np.cumsum(np.bincount(q, minlength=nq))]).astype(np.uint64)
    return offs, i[order].astype(np.uint64)


def count_path_reference(index, queries, coo, mode, thr):
    """Hits of a threshold >= 0 from the counts alone: containment count / |node| > thr, similarity (index without a
    num) count / (|node| + |query| - count) > thr; strict, per query by ascending index id."""
    assert thr >= 0.0
    q, i, c = coo
    den = index.lens[i].astype(np.float64)
    if mode == "similarity":
        den = (index.lens[i].astype(np.int64) + queries.lens[q].astype(np.int64) - c).astype(np.float64)
    return hits_from_cells(queries.n, q, i, c.astype(np.float64) / den > thr)


def assert_hits(got, want, what):
    offs, hits, total = got
    woffs, whits = want
    assert total == whits.size, f"{what}: {total} hits, want {whits.size}"
    assert np.array_equal(offs, woffs), f"{what}: per-query hit counts differ at queries {np.flatnonzero(np.diff(offs.astype(np.int64)) != np.diff(woffs.astype(np.int64)))[:10].tolist()}"
    assert np.array_equal(hits, whits), f"{what}: hit ids differ ({int(np.count_nonzero(hits != whits))} of {hits.size})"


@contextlib.contextmanager
def stream_launches():
    """Counts the launches of the index-streaming probe kernel inside the block: box[0] afterwards."""
    box = [0]
    smb.profile_enable(True)
    try:
        smb.profile_read("find_stream", reset=True)
        yield box
        box[0] = smb.profile_read("find_stream", reset=True)[1]
    finally:
        smb.profile_enable(False)


NQ = 2048
_search = {}


def search_case():
    """An index of scaled sketches (avg ~260 hashes) in clusters, and 2048 queries drawn from its clusters."""
    if not _search:
        index = Planted(70000, 0, SCALED_MAX_HASH, 0x5EA4C401, len_range=(20, 500), log_len=False, pool=700,
                        n_empty=6, n_single=6, extra_pool=200000)
        queries = Queries(index, related_queries(index, NQ, 0x5EA4C402))
        _search.update(index=index, queries=queries, coo=count_coo(index, queries))
    return _search["index"], _search["queries"], _search["coo"]


def assert_streams_automatically(index, queries):
    nq = queries.n
    assert index.n > FIND_BLOCK_CELLS // nq                              # two or more index blocks
    assert index.n_hashes >= STREAM_MIN_INDEX_HASHES                     # 'auto' streams ...
    assert index.n_hashes >= STREAM_INDEX_OVER_QUERY * queries.n_hashes  # ... this index past this batch
    assert index.n_hashes / index.n >= STREAM_MULTI_SLICE_AVG_LEN        # in more than one hash-range slice


# ------------------------------------------------------------------------------------------------
# (c) linear_find over several index blocks; the stream path chosen by 'auto'
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("thr", [0.0, 0.1, 0.6])
@pytest.mark.parametrize("mode", ["containment", "similarity"])
@pytest.mark.parametrize("path", ["auto", "join", "stream_small_spill"])
def test_find_multi_block(path, mode, thr):
    index, queries, coo = search_case()
    assert_streams_automatically(index, queries)
    want = count_path_reference(index, queries, coo, mode, thr)
    with knobs(find=path), stream_launches() as launches:
        got = find_raw(index.collection(), queries.collection(), mode, thr, want[1].size + 1)
    assert_hits(got, want, f"{path}/{mode}/{thr}")
    n_blocks = -(-index.n // (FIND_BLOCK_CELLS // queries.n))
    if path == "join":
        assert launches[0] == 0
    else:
        assert launches[0] >= n_blocks   # the index was streamed, block by block


@pytest.mark.parametrize("mode", ["containment", "similarity"])
def test_find_general_path_multi_block(mode):
    """threshold < 0: the f64 ratio matrix, the flags and their scan, over several blocks.  Every cell is a hit but
    those whose ratio is NaN (containment in an empty index sketch)."""
    index, queries, _ = search_case()
    assert index.n > FIND_BLOCK_CELLS // queries.n
    ids = np.arange(index.n, dtype=np.uint64)
    if mode == "containment":
        ids = ids[index.lens > 0]
        assert ids.size < index.n
    got = find_raw(index.collection(), queries.collection(), mode, -1.0, index.n * queries.n)
    offs, hits, total = got
    assert total == ids.size * queries.n
    assert np.array_equal(offs, np.arange(queries.n + 1, dtype=np.uint64) * np.uint64(ids.size))
    for q0 in range(0, queries.n, 256):
        blk = hits[q0 * ids.size:(q0 + 256) * ids.size].reshape(-1, ids.size)
        assert np.array_equal(blk, np.broadcast_to(ids, blk.shape)), f"queries {q0}..{q0 + 256}"


@pytest.mark.parametrize("thr", [0.0, 0.1])
def test_find_general_path_num_sketches(thr):
    """Similarity against an index of num sketches takes the general ratio path at every threshold; several blocks."""
    index = Planted(34000, 64, 0, 0x5EA4C411, full_len=64, extra_pool=20000)
    for k in (10, 11):   # shorter than num
        index.ids[k] = index.ids[k][:k - 5]
    index.lens = np.array([len(r) for r in index.ids], dtype=np.uint32)
    index.offsets = np.concatenate([[0], np.cumsum(index.lens, dtype=np.uint64)]).astype(np.uint64)
    index.hashes = index.values[np.concatenate(index.ids)]
    index.n_hashes = int(index.offsets[-1])
    queries = Queries(index, related_queries(index, 4096, 0x5EA4C412, num=64), num=64)
    assert index.n > FIND_BLOCK_CELLS // queries.n
    q, i, c = count_coo(index, queries)
    # KmerMinHash::compare(node, query) of every pair sharing a hash (the others have ratio 0)
    mhs = [index.oracle_sketch(k) for k in range(index.n)]
    for k in range(queries.n):
        o = orc.KmerMinHash(64, 31, False, 42, 0)
        o.add_many(queries.hashes[int(queries.offsets[k]):int(queries.offsets[k + 1])])
        mhs.append(o)
    oc, osz = orc.compare_pairs(mhs, i, q + index.n, NTHREADS)
    ratio = oc.astype(np.float64) / np.maximum(1, osz).astype(np.float64)
    want = hits_from_cells(queries.n, q, i, ratio > thr)
    got = find_raw(index.collection(), queries.collection(), "similarity", thr, want[1].size + 1)
    assert_hits(got, want, f"num sketches, similarity {thr}")


# ------------------------------------------------------------------------------------------------
# (d) searches in sequence on one context: the count matrix is cleared by the hit pass, never memset
# ------------------------------------------------------------------------------------------------
def test_find_searches_in_sequence():
    index, queries, coo = search_case()
    assert_streams_automatically(index, queries)
    icoll, qcoll = index.collection(), queries.collection()

    few = Queries(index, queries.ids[:100])
    small = Planted(30000, 0, SCALED_MAX_HASH, 0x5EA4C421, len_range=(20, 500), log_len=False, pool=700, n_empty=2)
    small_q = Queries(small, related_queries(small, 700, 0x5EA4C422))
    assert small.n_hashes >= max(STREAM_MIN_INDEX_HASHES, STREAM_INDEX_OVER_QUERY * small_q.n_hashes)
    steps = [
        ("first", index, icoll, queries, qcoll, coo, "containment", 0.1),
        ("100 queries", index, icoll, few, few.collection(), count_coo(index, few), "containment", 0.1),
        ("other index", small, small.collection(), small_q, small_q.collection(), count_coo(small, small_q), "similarity", 0.0),
        ("first again", index, icoll, queries, qcoll, coo, "containment", 0.1),
        ("first, similarity", index, icoll, queries, qcoll, coo, "similarity", 0.1),
    ]
    with stream_launches() as launches:
        for k, (what, ix, ic, qs, qc, cc, mode, thr) in enumerate(steps):
            if k == 3:   # a call refused by its compatibility check in between
                with pytest.raises(smb.SourmashError) as e:
                    smb.linear_find(ic, queries.collection(ksize=21), "containment", 0.1)
                assert e.value.code == 101
            want = count_path_reference(ix, qs, cc, mode, thr)
            assert_hits(find_raw(ic, qc, mode, thr, want[1].size + 1), want, what)
    assert launches[0] >= len(steps)   # every search streamed its index


# ------------------------------------------------------------------------------------------------
# (e) skewed query hashes: one table slice too large for shared memory, built in place
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", ["stream", "stream_small_spill", "join"])
def test_find_skewed_query_hashes(path):
    index, _, _ = search_case()
    top = int(index.hashes.max())
    low_limit = (top + 1) // QT_SLICES   # hashes below: table slice 0
    present = np.unique(np.concatenate(index.ids))
    low = present[index.values[present] < np.uint64(low_limit)]
    absent = index.extra[index.values[index.extra] < np.uint64(low_limit)]
    rng = np.random.Generator(np.random.PCG64(0x5EA4C431))
    ids = []
    for q in range(400):
        if q % 4 == 3:
            ids.append(ids[int(rng.integers(0, len(ids)))])   # duplicate queries
            continue
        r = np.unique(np.concatenate([rng.choice(low, 40, replace=False), rng.choice(absent, 3, replace=False)]))
        ids.append(r[np.argsort(index.values[r], kind="stable")])
    queries = Queries(index, ids)
    postings_slice0 = queries.n_hashes
    assert int(queries.hashes.max()) < low_limit
    assert 2 * postings_slice0 + 32 > QT_SMEM_SLOTS   # slice 0 does not fit shared memory
    coo = count_coo(index, queries)
    with knobs(find=path):
        for mode, thr in (("containment", 0.0), ("containment", 0.005), ("similarity", 0.0)):
            want = count_path_reference(index, queries, coo, mode, thr)
            assert want[1].size > 0
            got = find_raw(index.collection(), queries.collection(), mode, thr, want[1].size + 1)
            assert_hits(got, want, f"{path}/{mode}/{thr}")


# ------------------------------------------------------------------------------------------------
# (f) hash values with special handling: 0, 2^32 +- 1, 2^63 +- 1, 2^64 - 2 and 2^64 - 1 (the empty-slot key)
# ------------------------------------------------------------------------------------------------
def edge_rows(n, seed, row_len, shared=200):
    """Sorted unique rows: a random subset of the edge values (2^64 - 1 in most) and hashes from a shared pool."""
    rng = np.random.Generator(np.random.PCG64(seed))
    pool = np.setdiff1d(rng.integers(0, U64_MAX, size=shared, dtype=np.uint64, endpoint=True), EDGE)
    rows = []
    for k in range(n):
        length = row_len(rng) if callable(row_len) else row_len
        e = EDGE[rng.random(EDGE.size) < 0.5]
        if rng.random() < 0.7:
            e = np.union1d(e, EDGE[-1:])
        others = rng.permutation(pool[rng.random(pool.size) < 0.25])[:max(0, length - e.size)]
        r = np.union1d(e, others)
        if r.size > length:
            r = np.sort(r[rng.choice(r.size, length, replace=False)])
        rows.append(r)
    return rows


EDGE_KINDS = {
    # (num, max_hash, row lengths): full num sketches (dense rank kernel), short num sketches, scaled with max_hash 2^64 - 1
    "num_full": (16, 0, 16),
    "num": (64, 0, lambda rng: int(rng.integers(0, 49))),
    "scaled": (0, U64_MAX, lambda rng: int(rng.integers(0, 101))),
}
_edge = {}


def edge_case(kind):
    if kind not in _edge:
        num, mx, row_len = EDGE_KINDS[kind]
        rows = edge_rows(90, 0xED6E0000 + list(EDGE_KINDS).index(kind), row_len)
        rows[3] = rows[3][:0] if kind != "num_full" else rows[3]
        gs, os_ = [], []
        for r in rows:
            g = smb.KmerMinHash(num, 31, False, 42, mx)
            g.set_mins(r)
            o = orc.KmerMinHash(num, 31, False, 42, mx)
            o.add_many(r)
            assert np.array_equal(o.mins_np(), r)
            gs.append(g)
            os_.append(o)
        _edge[kind] = (rows, gs, os_)
    return _edge[kind]


@pytest.mark.parametrize("kind", list(EDGE_KINDS))
def test_edge_values_per_object(kind):
    rows, gs, os_ = edge_case(kind)
    num, mx, _ = EDGE_KINDS[kind]
    assert sum(int(r.size and r[-1] == EDGE[-1]) for r in rows) > 10
    for a in range(0, 30, 3):
        for b in (a, a + 1, a + 7, 89 - a):
            ga, gb, oa, ob = gs[a], gs[b], os_[a], os_[b]
            assert ga.count_common(gb) == oa.count_common(ob), (a, b)
            assert ga.compare(gb) == oa.compare(ob), (a, b)
            gi, gsz = ga.intersection(gb)
            oi, osz = oa.intersection(ob)
            assert np.array_equal(gi, oi) and gsz == osz, (a, b)
            gc, oc = ga.containment(gb), oa.containment(ob)
            assert gc == oc or (np.isnan(gc) and np.isnan(oc)), (a, b)
            gm, om = smb.KmerMinHash(num, 31, False, 42, mx), orc.KmerMinHash(num, 31, False, 42, mx)
            gm.set_mins(rows[a])
            om.add_many(rows[a])
            gm.merge(gb)
            om.merge(ob)
            assert np.array_equal(gm.mins_np(), om.mins_np()), (a, b)


@pytest.mark.parametrize("abund", [False, True])
def test_edge_values_add_many(abund):
    """Batches with every edge value (repeated) into a scaled sketch with max_hash 2^64 - 1 and into a num sketch:
    new hashes fold through the one-CTA sort (at most FOLD_SMALL of them) or through the generic union."""
    rng = np.random.Generator(np.random.PCG64(0xED6E0100 + abund))
    pool = rng.integers(0, U64_MAX, size=20000, dtype=np.uint64, endpoint=True)
    for num, mx in ((0, U64_MAX), (300, 0)):
        g, o = smb.KmerMinHash(num, 31, False, 42, mx, abund), orc.KmerMinHash(num, 31, False, 42, mx, abund)
        cursor = 0
        for n_new, with_edge in ((3000, False), (100, True), (FOLD_SMALL - 20, True), (3 * FOLD_SMALL, True), (5, True)):
            fresh = pool[cursor:cursor + n_new]
            cursor += n_new
            batch = np.concatenate([fresh, EDGE, EDGE[-3:], pool[:cursor - n_new:50]]) if with_edge else fresh
            batch = batch[rng.permutation(batch.size)]
            g.add_many(batch)
            o.add_many(batch)
            assert np.array_equal(g.mins_np(), o.mins_np()), (num, n_new)
            if abund:
                assert np.array_equal(g.abunds_np(), o.abunds_np()), (num, n_new)
        if num == 0:
            assert g.mins_np()[-1] == EDGE[-1] and g.mins_np()[0] == 0


@pytest.mark.parametrize("path", ["auto", "sparse", "dense"])
@pytest.mark.parametrize("kind", list(EDGE_KINDS))
def test_edge_values_compare_matrix(kind, path):
    rows, gs, os_ = edge_case(kind)
    coll = smb.SketchCollection.from_sketches(gs)
    oc, osz = orc.compare_matrix(os_, os_)
    occ = orc.count_common_matrix(os_, os_)
    lens = np.array([r.size for r in rows], dtype=np.uint32)
    with knobs(compare=path):
        common, size, ratio = smb.compare_matrix(coll, coll, "compare")
        assert not mismatch("common", common, oc) and not mismatch("size", size, osz)
        assert not mismatch("ratio", ratio, oc / np.maximum(1, osz).astype(np.float64))
        common, size, ratio = smb.compare_matrix(coll, coll, "containment")
        assert not mismatch("containment common", common, occ)
        assert np.array_equal(size, np.repeat(lens[:, None], lens.size, 1))
        with np.errstate(invalid="ignore"):
            assert not mismatch("containment ratio", ratio, occ / np.repeat(lens[:, None], lens.size, 1).astype(np.float64))
        part = smb.SketchCollection.from_sketches(gs[20:45])   # two collections: postings of both sides
        common, size, ratio = smb.compare_matrix(part, coll, "compare")
        assert not mismatch("two collections", common, oc[20:45]) and not mismatch("two collections size", size, osz[20:45])


@pytest.mark.parametrize("path", ["stream", "stream_small_spill", "join"])
@pytest.mark.parametrize("kind", list(EDGE_KINDS))
def test_edge_values_linear_find(kind, path):
    rows, gs, os_ = edge_case(kind)
    index = smb.SketchCollection.from_sketches(gs)
    qsel = list(range(0, 90, 4))
    assert sum(int(rows[q].size and rows[q][-1] == EDGE[-1]) for q in qsel) > 3   # several nodes on the 2^64 - 1 list
    assert max(int(r[-1]) for r in rows if r.size) == U64_MAX                        # the index top is 2^64 - 1
    queries = smb.SketchCollection.from_sketches([gs[q] for q in qsel])
    modes = ["containment"] + (["similarity"] if kind == "scaled" else [])
    with knobs(find=path), stream_launches() as launches:
        for mode in modes:
            for thr in (0.0, 0.1, 0.5):
                got = smb.linear_find(index, queries, mode, thr)
                for k, q in enumerate(qsel):
                    assert got[k] == orc.linear_find(os_, os_[q], mode, thr), (mode, thr, q)
    assert (launches[0] > 0) == (path != "join")


@pytest.mark.parametrize("kind", list(EDGE_KINDS))
def test_edge_values_scaffold_pairs(kind):
    rows, gs, os_ = edge_case(kind)
    for n in (90, 41):
        assert smb.scaffold_pairs(smb.SketchCollection.from_sketches(gs[:n])) == orc.scaffold_pairs(os_[:n])
