"""Round-2 additions, each against the CPU oracle through the C ABI:
  * KmerMinHash::intersection returning the hashes (lib.rs:438-468), the jaccard / containment C names;
  * the estimate-threshold acceptance rule of num sketches that are only partly full;
  * host threads: distinct handles driven concurrently (SURVEY 8(b) Threading, utils.rs:14-16), a handle
    moving between threads, concurrent readers of one handle."""
import threading

import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from util import MAX_HASH_1000, golden, make_reads, mutate, random_dna

pytestmark = pytest.mark.gpu


def _same(g, o, ctx=None):
    assert np.array_equal(g.mins_np(), o.mins_np()), ctx
    ga, oa = g.abunds_np(), o.abunds_np()
    assert (ga is None) == (oa is None), ctx
    if ga is not None:
        assert np.array_equal(ga, oa), ctx


def _pair(num, k, mx=0, ab=False):
    return smb.KmerMinHash(num, k, False, 42, mx, ab), orc.KmerMinHash(num, k, False, 42, mx, ab)


# ------------------------------------------------------------------------------------------------
# intersection (hashes), jaccard, containment
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("num,mx", [(500, 0), (50, 0), (0, MAX_HASH_1000 * 10), (0, 0), (200, MAX_HASH_1000 * 100)])
def test_intersection_hashes_and_names(num, mx):
    g0 = random_dna(60_000, 31)
    g1 = mutate(g0, 0.02, 32)
    a, oa = _pair(num, 21, mx)
    b, ob = _pair(num, 21, mx)
    a.add_sequence(g0); oa.add_sequence(g0)
    b.add_sequence(g1); ob.add_sequence(g1)
    for x, y, ox, oy in ((a, b, oa, ob), (b, a, ob, oa), (a, a, oa, oa)):
        hashes, size = x.intersection(y)
        ohashes, osize = ox.intersection(oy)
        assert size == osize and np.array_equal(hashes, ohashes)
        assert (len(hashes), size) == ox.intersection_size(oy)
        assert x.jaccard(y) == ox.compare(oy) == x.compare(y)
        c, oc = x.containment(y), ox.containment(oy)
        assert c == oc or (np.isnan(c) and np.isnan(oc))
    e, oe = _pair(num, 21, mx)
    hashes, size = a.intersection(e)
    assert len(hashes) == 0 and size == oa.intersection(oe)[1]
    assert np.isnan(e.containment(a)) and np.isnan(oe.containment(oa))   # 0/0 (index.rs:152-154)
    other_k = smb.KmerMinHash(num, 31, False, 42, mx)
    for f in (a.jaccard, a.containment, a.intersection):
        with pytest.raises(smb.SourmashError) as err:
            f(other_k)
        assert err.value.code == 101


def test_intersection_hashes_on_the_reference_fixture():  # the (common, size) matrix SURVEY 8(c) lists
    g = golden("sbt_v5_leaves.json")
    mhs, omhs = [], []
    for p in sorted(g["leaves"], key=int):           # tree positions 6..12
        sk = g["leaves"][p]["sketch"]
        m = smb.KmerMinHash(sk["num"], sk["ksize"], False, sk["seed"], sk["max_hash"])
        m.set_mins(sk["mins"])
        mhs.append(m)
        om = orc.KmerMinHash(sk["num"], sk["ksize"], False, sk["seed"], sk["max_hash"])
        for h in sk["mins"]:
            om.mins_push(h)
        omhs.append(om)
    assert np.array_equal(mhs[1].intersection(mhs[5])[0], omhs[1].intersection(omhs[5])[0])
    hashes, size = mhs[1].intersection(mhs[5])       # leaves 7 and 11: Jaccard 178/500
    assert (len(hashes), size) == (178, 500)
    assert np.all(np.diff(hashes.astype(np.uint64)) > 0)
    assert set(hashes.tolist()) <= (set(mhs[1].mins_np().tolist()) & set(mhs[5].mins_np().tolist()))
    assert mhs[1].containment(mhs[5]) == 268 / 500


# ------------------------------------------------------------------------------------------------
# partly full num sketch + a long sequence whose windows are mostly unusable: the estimated kernel
# threshold keeps too few hashes, and elements of the old state above it must not make that look like enough
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("abund", [False, True])
@pytest.mark.parametrize("kind", ["mostly_n", "tandem"])
def test_partly_full_num_sketch_then_low_yield_long_sequence(abund, kind):
    num, k = 500, 21
    g, o = _pair(num, k, 0, abund)
    short = random_dna(260, 5)            # 240 hashes: fewer than num
    g.add_sequence(short); o.add_sequence(short)
    assert 0 < g.size() < num
    if kind == "mostly_n":
        body = bytearray(b"N" * 400_000)
        island = random_dna(3000, 6)      # ~2 980 valid windows in 400 kbp
        for i in range(0, 3000, 100):
            pos = 1000 + i * 130
            body[pos:pos + 100] = island[i:i + 100]
        long_seq = bytes(body)
    else:
        long_seq = random_dna(700, 7) * 300   # 210 kbp, 700 distinct windows
    g.add_sequence(long_seq, True); o.add_sequence(long_seq, True)
    _same(g, o)
    g.add_sequence(random_dna(50_000, 8)); o.add_sequence(random_dna(50_000, 8))
    _same(g, o)


# ------------------------------------------------------------------------------------------------
# host threads
# ------------------------------------------------------------------------------------------------
def test_distinct_handles_on_distinct_threads():
    n_threads = 8
    genome = random_dna(400_000, 77)
    reads = [make_reads(genome, 3000, 150, 100 + t) for t in range(n_threads)]
    big = [random_dna(300_000, 200 + t) for t in range(n_threads)]
    results, errors = [None] * n_threads, []

    def work(t):
        try:
            a = smb.KmerMinHash(0, 31, False, 42, MAX_HASH_1000 * 10, True)
            b = smb.KmerMinHash(300, 21, False, 42, 0, t % 2 == 0)
            rd = reads[t]
            for i in range(0, len(rd), 150):            # the reference's calling pattern: one read per call
                a.add_sequence(rd[i:i + 150])
            for i in range(0, len(rd) // 2, 150):
                b.add_sequence(rd[i:i + 150])
            a.add_sequence(big[t]); b.add_sequence(big[t])  # the synchronous path
            a.add_reads(rd, len(rd) // 150, 150)            # and the batch entry point
            sig = smb.Signature()
            sig.push_mh(a)
            results[t] = (a.mins_np(), a.abunds_np(), b.mins_np(), b.abunds_np(), a.compare(a), a.count_common(a),
                          sig.save_json())
        except Exception as e:  # noqa: BLE001
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=work, args=(t,)) for t in range(n_threads)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    for t in range(n_threads):
        oa = orc.KmerMinHash(0, 31, False, 42, MAX_HASH_1000 * 10, True)
        ob = orc.KmerMinHash(300, 21, False, 42, 0, t % 2 == 0)
        rd = reads[t]
        oa.add_reads(rd, len(rd) // 150, 150)
        ob.add_reads(rd[:225_000], 1500, 150)              # the reads starting below len(rd) // 2
        oa.add_sequence(big[t]); ob.add_sequence(big[t])
        oa.add_reads(rd, len(rd) // 150, 150)
        am, aa, bm, ba, cmp_, cc, js = results[t]
        assert np.array_equal(am, oa.mins_np()) and np.array_equal(aa, oa.abunds_np()), t
        assert np.array_equal(bm, ob.mins_np()), t
        if ba is not None:
            assert np.array_equal(ba, ob.abunds_np()), t
        assert cmp_ == 1.0 and cc == oa.size()
        assert js == orc.signature_json([oa])


def test_a_handle_moves_between_threads():
    g, o = _pair(0, 21, MAX_HASH_1000 * 20, True)
    chunks = [random_dna(120_000, 300 + i) for i in range(6)]
    coll_holder = {}

    def step(i):
        g.add_sequence(chunks[i])                       # device work queued from this thread ...
        for j in range(0, 3000, 150):
            g.add_sequence(chunks[i][j:j + 150])        # ... and deferred reads left pending on the handle
        if i == 3:
            coll_holder["c"] = smb.SketchCollection.from_sketches([g])

    for i in range(6):
        th = threading.Thread(target=step, args=(i,))
        th.start(); th.join()
        o.add_sequence(chunks[i])
        for j in range(0, 3000, 150):
            o.add_sequence(chunks[i][j:j + 150])
        if i == 3:
            snap = o.mins_np()
    _same(g, o)                                         # read on the main thread
    assert np.array_equal(coll_holder["c"].rows_np()[0], snap)
    common, size, ratio = smb.compare_matrix(coll_holder["c"], coll_holder["c"])   # a collection built on a thread that is gone
    assert common[0, 0] == size[0, 0] == len(snap) and ratio[0, 0] == 1.0


def test_concurrent_readers_of_one_handle():
    a, oa = _pair(0, 31, MAX_HASH_1000 * 10, False)
    b, ob = _pair(0, 31, MAX_HASH_1000 * 10, False)
    g0 = random_dna(500_000, 41)
    g1 = mutate(g0, 0.01, 42)
    a.add_sequence(g0); oa.add_sequence(g0)
    for i in range(0, len(g1) - 1000, 1000):            # b is left with deferred reads: the first reader flushes them
        b.add_sequence(g1[i:i + 1030]); ob.add_sequence(g1[i:i + 1030])
    want = (oa.compare(ob), oa.count_common(ob), ob.size())
    got, errors = [], []

    def reader():
        try:
            for _ in range(20):
                got.append((a.compare(b), a.count_common(b), b.size()))
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))

    threads = [threading.Thread(target=reader) for _ in range(6)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors
    assert len(got) == 120 and all(x == want for x in got)


# ------------------------------------------------------------------------------------------------
# linear_find over a large index: the streaming path (csrc/find_stream.cu) against the oracle and the join path
# ------------------------------------------------------------------------------------------------
def _index_and_queries(n_index, n_q, lens, mx, num, seed, dup_queries=True):
    r = np.random.Generator(np.random.PCG64(seed))
    hi = mx if mx else 1 << 60
    base = [np.unique(r.integers(0, hi, size=lens[1], dtype=np.uint64)) for _ in range(max(2, n_index // 20))]
    rows = []
    for i in range(n_index):
        b = base[i % len(base)]
        keep = b[r.random(b.size) < (0.05, 0.3, 0.6, 0.95)[i % 4]]
        row = np.unique(np.concatenate([keep, r.integers(0, hi, size=int(r.integers(lens[0], lens[1])), dtype=np.uint64)]))
        rows.append(row[:num] if num else row)
    rows[1] = rows[1][:0]                      # an empty index sketch (containment 0/0 = NaN: never a hit)
    rows[2] = rows[2][:3]
    queries = []
    for q in range(n_q):
        row = np.unique(np.concatenate([base[q % len(base)][::2], r.integers(0, hi, size=int(r.integers(1, lens[1])), dtype=np.uint64)]))
        queries.append(row[:num] if num else row)
    if dup_queries and n_q > 3:
        queries[3] = queries[0].copy()         # the same hashes in two queries: table runs longer than one
        queries[2] = queries[2][:0]            # an empty query
    return rows, queries


def _colls(rows, num, mx):
    g, o = [], []
    for row in rows:
        a, b = smb.KmerMinHash(num, 31, False, 42, mx), orc.KmerMinHash(num, 31, False, 42, mx)
        a.set_mins(row); b.add_many(row)
        g.append(a); o.append(b)
    return smb.SketchCollection.from_sketches(g), o


@pytest.mark.parametrize("n_index,n_q,lens,mx,num", [
    (300, 12, (50, 2500), MAX_HASH_1000 * 4, 0),        # ragged scaled sketches, few slices
    (150, 9, (7000, 9000), MAX_HASH_1000 * 8, 0),       # long sketches: 64 slices, stretches above and below 96 hashes
    (5000, 6, (100, 400), MAX_HASH_1000, 0),            # more rows than one chunk of a work item
    (400, 10, (300, 900), 0, 500),                      # num sketches (containment only decides by count)
    (40, 40, (5, 60), MAX_HASH_1000, 0),                # tiny rows, as many queries as index sketches
])
def test_linear_find_streaming_path(n_index, n_q, lens, mx, num):
    rows, queries = _index_and_queries(n_index, n_q, lens, mx, num, 1000 + n_index)
    ic, o_index = _colls(rows, num, mx)
    qc, o_queries = _colls(queries, num, mx)
    try:
        n_hits = 0
        for mode in ("containment", "similarity"):
            for thr in (0.0, 0.1, 0.6):
                smb.find_path("join")
                want = smb.linear_find(ic, qc, mode, thr)
                smb.find_path("stream")
                got = smb.linear_find(ic, qc, mode, thr)
                assert got == want, (mode, thr)
                smb.find_path("stream_small_spill")   # the written-out hits overflow: the block runs again, lookups in the kernel
                assert smb.linear_find(ic, qc, mode, thr) == want, (mode, thr, "small spill")
                smb.find_path("stream")
                n_hits += sum(len(h) for h in got)
                for q in range(0, n_q, max(1, n_q // 4)):
                    assert got[q] == orc.linear_find(o_index, o_queries[q], mode, thr), (mode, thr, q)
        assert n_hits > 0
        # the index changes: the slice bounds kept with it are rebuilt
        extra = smb.KmerMinHash(num, 31, False, 42, mx)
        extra.set_mins(queries[0])
        ic.push(extra)
        got = smb.linear_find(ic, qc, "containment", 0.5)
        assert n_index in got[0] and (len(queries[3]) == 0 or n_index in got[3])
    finally:
        smb.find_path("auto")


# ------------------------------------------------------------------------------------------------
# merge of a sketch whose abundances are out of step with its mins (the state lib.rs:395-400 leaves behind)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("track", [(True, True, True), (True, False, True), (False, True, True), (True, True, False)])
def test_chained_merges_after_truncation(track):
    num, k = 150, 21
    seqs = [random_dna(4000, 900 + i) + random_dna(3000, 950) for i in range(3)]   # a shared stretch: common hashes
    gs = [smb.KmerMinHash(num, k, False, 42, 0, t) for t in track]
    os_ = [orc.KmerMinHash(num, k, False, 42, 0, t) for t in track]
    for g, o, s in zip(gs, os_, seqs):
        g.add_sequence(s); o.add_sequence(s)
        g.add_sequence(s[:2000]); o.add_sequence(s[:2000])       # abundances above 1
    gs[0].merge(gs[1]); os_[0].merge(os_[1])                      # mins truncated to num, abundances not
    _same(gs[0], os_[0], "first merge")
    assert len(gs[0].abunds_np()) != gs[0].size() or not (track[0] and track[1])
    gs[0].merge(gs[2]); os_[0].merge(os_[2])                      # ... and merged again: walked step by step
    _same(gs[0], os_[0], "second merge")
    gs[2].merge(gs[0]); os_[2].merge(os_[0])                      # the out-of-step sketch on the other side
    _same(gs[2], os_[2], "third merge")
    gs[0].merge(gs[0].__class__(num, k, False, 42, 0, True)); os_[0].merge(orc.KmerMinHash(num, k, False, 42, 0, True))  # with an empty one
    _same(gs[0], os_[0], "merge with empty")


def test_host_threads_add_up():
    """Eight host threads, each feeding its own sketch through the unmodified kmerminhash_add_sequence (a C loop,
    host/feed_reads.c), against one thread feeding the same reads: no library-wide lock, so the aggregate rate
    must go up (it is host-bound: validation + staging of each read), and every thread's sketch must be right."""
    n, L = 1_600_000, 150     # 30 MB per thread: several 8 MiB flushes each
    genome = random_dna(1_000_000, 5)
    reads = np.frombuffer(make_reads(genome, n, L, 6), dtype=np.uint8).reshape(n, L)
    z = np.zeros((n, L + 1), dtype=np.uint8)
    z[:, :L] = reads

    def run(threads):
        groups = [[smb.KmerMinHash(0, 31, False, 42, MAX_HASH_1000, True)] for _ in range(threads)]
        secs = smb.feed_reads(groups, z, n, L + 1, warm_reads=10_000)
        return (n - 10_000 * threads) * L / secs, groups

    run(8)                    # first use: page-locked staging buffers, per-thread scratch
    rate1, g1 = run(1)
    rate8, g8 = run(8)
    print("aggregate Gbp/s: 1 thread %.2f, 8 threads %.2f" % (rate1 / 1e9, rate8 / 1e9))
    assert rate8 > 1.3 * rate1, (rate1, rate8)
    # parity: thread t fed reads [t * n / 8, (t + 1) * n / 8)
    per = n // 8
    for t in (0, 3, 7):
        o = orc.KmerMinHash(0, 31, False, 42, MAX_HASH_1000, True)
        o.add_reads(reads[t * per:(t + 1) * per].tobytes(), per, L)
        _same(g8[t][0], o, t)
    o = orc.KmerMinHash(0, 31, False, 42, MAX_HASH_1000, True)
    o.add_reads(reads.tobytes(), n, L)
    _same(g1[0][0], o)


# ------------------------------------------------------------------------------------------------
# the sparse path's pair walk over short sketches, num sketches cut below num, and a row shard, against the oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("num,lens", [(400, (400, 401)), (0, (0, 500)), (100, (30, 300)), (512, (512, 513))])
def test_sparse_walk_over_short_and_partial_num_sketches(num, lens):
    r = np.random.Generator(np.random.PCG64(num + 17))
    base = [np.unique(r.integers(0, 1 << 60, size=700, dtype=np.uint64)) for _ in range(6)]
    rows, g_sk, o_sk = [], [], []
    for i in range(150):
        b = base[i % 6]
        keep = b[r.random(b.size) < (0.2, 0.6, 0.95)[i % 3]]
        row = np.unique(np.concatenate([keep, r.integers(0, 1 << 60, size=200, dtype=np.uint64)]))
        row = row[: int(r.integers(lens[0], lens[1]))]
        if num and i % 7 == 0:
            row = row[: num // 3]                   # not full: the union may hold fewer than num elements
        rows.append(row)
        mx = 0 if num else 1 << 60                  # (num = 0 needs a max_hash: scaled sketches)
        g, o = smb.KmerMinHash(num, 31, False, 42, mx), orc.KmerMinHash(num, 31, False, 42, mx)
        g.set_mins(row); o.add_many(row)
        g_sk.append(g); o_sk.append(o)
    coll = smb.SketchCollection.from_sketches(g_sk)
    part = smb.SketchCollection.from_sketches(g_sk[20:60])
    oc, osz = orc.compare_matrix(o_sk, o_sk)
    try:
        smb.compare_path("sparse")
        common, size, ratio = smb.compare_matrix(coll, coll)             # the whole square: each unordered pair once
        assert np.array_equal(common, oc) and np.array_equal(size, osz)
        assert np.array_equal(ratio, oc.astype(np.float64) / np.maximum(1, osz).astype(np.float64))
        common, size, _ = smb.compare_matrix(part, coll)                 # a row shard against everything
        assert np.array_equal(common, oc[20:60]) and np.array_equal(size, osz[20:60])
    finally:
        smb.compare_path("auto")


# ------------------------------------------------------------------------------------------------
# 2-bit packed reads (an input format of this build, not of the reference): same sketches as the ASCII form
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_reads,read_len", [(120_000, 150), (5000, 151), (3000, 64), (7, 33), (1, 21)])
def test_packed_2bit_reads_equal_ascii(n_reads, read_len):
    genome = random_dna(max(400_000, 4 * read_len), 60 + read_len)
    reads = np.frombuffer(make_reads(genome, n_reads, read_len, 61), dtype=np.uint8).reshape(n_reads, read_len)
    packed = smb.pack_2bit(reads, read_len)
    assert packed.shape == (n_reads, (read_len + 3) // 4)
    ks = [k for k in (21, 31, 51) if k <= read_len]
    want = [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000 * 5, True) for k in ks]
    smb.add_reads(want, reads.tobytes(), n_reads, read_len)
    got = [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000 * 5, True) for k in ks]
    smb.add_reads_2bit(got, packed, n_reads, read_len)                      # host buffer: chunks cross PCIe packed
    for g, w in zip(got, want):
        assert np.array_equal(g.mins_np(), w.mins_np()) and np.array_equal(g.abunds_np(), w.abunds_np())
    o = orc.KmerMinHash(0, ks[0], False, 42, MAX_HASH_1000 * 5, True)
    o.add_reads(reads[:20_000].tobytes(), min(n_reads, 20_000), read_len)
    chk = smb.KmerMinHash(0, ks[0], False, 42, MAX_HASH_1000 * 5, True)
    smb.add_reads_2bit([chk], packed[:20_000], min(n_reads, 20_000), read_len)
    _same(chk, o)
    import torch                                                             # packed reads already in HBM
    dev_packed = torch.from_numpy(packed.copy()).cuda()
    num_sk = smb.KmerMinHash(300, ks[0], False, 42, 0, True)
    num_ref = smb.KmerMinHash(300, ks[0], False, 42, 0, True)
    smb.add_reads_2bit([num_sk], dev_packed.data_ptr(), n_reads, read_len, on_device=True)
    smb.add_reads([num_ref], reads.tobytes(), n_reads, read_len)
    assert np.array_equal(num_sk.mins_np(), num_ref.mins_np()) and np.array_equal(num_sk.abunds_np(), num_ref.abunds_np())
