"""GPU parity tests: every result that comes out of the C ABI (include/sourmash.h and
include/sourmash_b200.h) is compared bit-for-bit with the CPU oracle (oracle/oracle.c, a
restatement of the reference pinned by tests/test_oracle.py) on the same inputs, and with the
reference's own known-answer tests and fixtures."""
import contextlib
import json

import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from util import MAX_HASH_1000, golden, make_reads, mutate, random_dna, splitmix64

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


def pair(num, k, max_hash=0, abund=False, seed=42):
    return smb.KmerMinHash(num, k, False, seed, max_hash, abund), orc.KmerMinHash(num, k, False, seed, max_hash, abund)


def same(g, o):
    assert np.array_equal(g.mins_np(), o.mins_np()), (g.mins_np()[:5], o.mins_np()[:5], g.size(), o.size())
    ga, oa = g.abunds_np(), o.abunds_np()
    assert (ga is None) == (oa is None)
    if ga is not None:
        assert np.array_equal(ga, oa)


def dirty(seq: bytes, seed, n_bad=12, lower=True):
    """sprinkle lower-case stretches and invalid bytes"""
    a = bytearray(seq)
    r = splitmix64(seed, n_bad * 2 + 8)
    if lower:
        for i in range(4):
            s = int(r[i] % np.uint64(max(1, len(a) - 50)))
            a[s:s + 40] = bytes(a[s:s + 40]).lower()
    for i in range(n_bad):
        a[int(r[8 + i] % np.uint64(len(a)))] = b"NRYn-*"[int(r[8 + n_bad + i] % np.uint64(6))]
    return bytes(a)


# ------------------------------------------------------------------------------------------------
# the reference's own tests, through the C ABI
# ------------------------------------------------------------------------------------------------
def test_throws_error():  # tests/minhash.rs:5-17
    mh = smb.KmerMinHash(1, 4)
    with pytest.raises(smb.SourmashError) as e:
        mh.add_sequence(b"ATGR", False)
    assert e.value.code == 1101
    assert e.value.message == "invalid DNA character in input k-mer: ATGR"


def test_merge_kat():  # tests/minhash.rs:19-52
    a, b = smb.KmerMinHash(20, 10), smb.KmerMinHash(20, 10)
    a.add_sequence(b"TGCCGCCCAGCA"); b.add_sequence(b"TGCCGCCCAGCA")
    a.add_sequence(b"GTCCGCCCAGTGA"); b.add_sequence(b"GTCCGCCCAGTGG")
    a.merge(b)
    assert a.mins == [2996412506971915891, 4448613756639084635, 8373222269469409550, 9390240264282449587,
                      11085758717695534616, 11668188995231815419, 11760449009842383350, 14682565545778736889]
    assert a.track_abundance() and a.abunds == []  # lib.rs:393


def test_compare_kat():  # tests/minhash.rs:54-83
    s1 = b"TGCCGCCCAGCACCGGGTGACTAGGTTGAGCCATGATTAACCTGCAATGA"
    s2 = b"GATTGGTGCACACTTAACTGGGTGCCGCGCTGGTGCTGATCCATGAAGTT"
    a, b = smb.KmerMinHash(20, 10), smb.KmerMinHash(20, 10)
    a.add_sequence(s1); b.add_sequence(s1)
    assert a.compare(b) == 1.0 and b.compare(a) == 1.0
    b.add_sequence(s1)
    assert a.compare(b) == 1.0 and b.compare(a) == 1.0
    b.add_sequence(s2)
    assert a.compare(b) >= 0.3 and b.compare(a) >= 0.3
    oa, ob = orc.KmerMinHash(20, 10), orc.KmerMinHash(20, 10)
    oa.add_sequence(s1); ob.add_sequence(s1); ob.add_sequence(s1); ob.add_sequence(s2)
    assert a.compare(b) == oa.compare(ob) and b.compare(a) == ob.compare(oa)


def _load(mod, sk):
    mh = mod.KmerMinHash(0 if sk["max_hash"] else sk["num"], sk["ksize"], sk["molecule"] == "protein", sk["seed"],
                         sk["max_hash"], "abundances" in sk)
    for m in sk["mins"]:
        mh.mins_push(m)
    for a in sk.get("abundances", []):
        mh.abunds_push(a)
    return mh


V5_COMPARE = [[500, 43, 0, 37, 0, 39, 0], [43, 500, 0, 39, 0, 178, 0], [0, 0, 500, 0, 191, 0, 182],
              [37, 39, 0, 500, 0, 36, 0], [0, 0, 191, 0, 500, 0, 193], [39, 178, 0, 36, 0, 500, 0],
              [0, 0, 182, 0, 193, 0, 500]]
V5_COMMON = [[500, 54, 0, 61, 0, 55, 0], [54, 500, 0, 70, 0, 268, 0], [0, 0, 500, 0, 267, 0, 275],
             [61, 70, 0, 500, 0, 68, 0], [0, 0, 267, 0, 500, 0, 273], [55, 268, 0, 68, 0, 500, 0],
             [0, 0, 275, 0, 273, 0, 500]]


def test_sbt_v5_fixture_pairs_and_search():  # src/index/sbt.rs:543-588 + SURVEY 8(c) golden integers
    g = golden("sbt_v5_leaves.json")
    pos = sorted(g["leaves"], key=int)
    leaves = [_load(smb, g["leaves"][p]["sketch"]) for p in pos]
    # per-object ABI
    for i in range(7):
        for j in range(7):
            assert leaves[i].count_common(leaves[j]) == V5_COMMON[i][j]
            assert leaves[i].compare(leaves[j]) == V5_COMPARE[i][j] / 500
            assert leaves[i].intersection_union_size(leaves[j]) == 500
    # collection kernels
    coll = smb.SketchCollection.from_sketches(leaves)
    common, size, ratio = smb.compare_matrix(coll, coll, "compare")
    assert common.tolist() == V5_COMPARE and (size == 500).all()
    assert np.array_equal(ratio, np.array(V5_COMPARE, dtype=np.float64) / 500.0)
    common, size, ratio = smb.compare_matrix(coll, coll, "containment")
    assert common.tolist() == V5_COMMON and (size == 500).all()
    q = smb.SketchCollection.from_sketches([leaves[pos.index(g["query_position"])]])
    want = g["asserted_hits"]
    for mode in ("similarity", "containment"):
        for thr in (0.5, 0.1):
            hits = smb.linear_find(coll, q, mode, thr)[0]
            assert len(hits) == want["%s@%s" % (mode, thr)]
    assert [int(pos[i]) for i in smb.linear_find(coll, q, "similarity", 0.1)[0]] == [7, 11]
    assert [int(pos[i]) for i in smb.linear_find(coll, q, "containment", 0.1)[0]] == [6, 7, 9, 11]


def test_md5sum_fixtures():  # lib.rs:72-77
    g = golden("sbt_v5_leaves.json")
    for leaf in g["leaves"].values():
        assert _load(smb, leaf["sketch"]).md5sum() == leaf["sketch"]["md5sum"]
    for sk in golden("genome_s10_s11.json")["sketches"]:
        assert _load(smb, sk).md5sum() == sk["md5sum"]


# ------------------------------------------------------------------------------------------------
# add_sequence: GPU sketch kernel vs oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [21, 31, 51, 4, 10, 32, 33, 64, 70])
@pytest.mark.parametrize("kind", ["num", "scaled", "num_abund", "scaled_abund"])
def test_add_sequence_parity(k, kind):
    seq = dirty(random_dna(60000, 0x5EED0001 + k), 77 + k)
    num = 500 if kind.startswith("num") else 0
    mx = 0 if kind.startswith("num") else MAX_HASH_1000 * 20
    g, o = pair(num, k, mx, kind.endswith("abund"))
    g.add_sequence(seq, True); o.add_sequence(seq, True)
    same(g, o)
    # a second call on top of the existing state (repeats -> abundances, threshold from the state)
    seq2 = seq[10000:30000] + random_dna(5000, 99)
    g.add_sequence(seq2, True); o.add_sequence(seq2, True)
    same(g, o)


@pytest.mark.parametrize("k", [21, 31, 51])
def test_large_genome_num500(k):  # BASELINE config 1 shape at reduced length for the oracle
    g0 = random_dna(1_000_000, 0x5EED0001)
    g1 = mutate(g0, 0.01, 0x5EED0002)
    a, oa = pair(500, k)
    b, ob = pair(500, k)
    a.add_sequence(g0); oa.add_sequence(g0)
    b.add_sequence(g1); ob.add_sequence(g1)
    same(a, oa); same(b, ob)
    assert a.compare(b) == oa.compare(ob)
    assert a.count_common(b) == oa.count_common(ob)


def test_repetitive_sequence_num():  # few distinct k-mers: the threshold estimate must widen
    seq = (b"ACGTTGCAAC" * 30000)
    g, o = pair(500, 21, 0, True)
    g.add_sequence(seq); o.add_sequence(seq)
    same(g, o)
    g2, o2 = pair(5, 21, 0, True)
    g2.add_sequence(seq); o2.add_sequence(seq)
    same(g2, o2)


def test_force_false_partial_state_and_message():
    seq = bytearray(random_dna(9000, 5))
    seq[7000] = ord("N")
    seq = bytes(seq)
    for k, num, mx in ((21, 50, 0), (31, 0, MAX_HASH_1000 * 100), (10, 30, 0)):
        g, o = pair(num, k, mx, True)
        with pytest.raises(smb.SourmashError) as ge:
            g.add_sequence(seq, False)
        with pytest.raises(orc.SourmashError) as oe:
            o.add_sequence(seq, False)
        assert ge.value.code == oe.value.code == 1101
        assert ge.value.message == oe.value.message
        same(g, o)
    # lower-case input: the k-mer in the message is upper-cased (lib.rs:253-256)
    g, o = pair(10, 5)
    with pytest.raises(smb.SourmashError) as ge:
        g.add_sequence(b"acgtacgtnacgt", False)
    with pytest.raises(orc.SourmashError) as oe:
        o.add_sequence(b"acgtacgtnacgt", False)
    assert ge.value.message == oe.value.message
    same(g, o)


def test_short_and_edge_sequences():
    for seq in (b"", b"A", b"ACG", b"ACGTA", b"ACGTAC", b"NNNNNNNN", b"ACGTN", b"NACGTA"):
        g, o = pair(10, 5, 0, True)
        g.add_sequence(seq, True); o.add_sequence(seq, True)
        same(g, o)
    # around the tile size (4096 window starts per tile) and its multiples
    for n in (2047, 2048, 2049, 4095, 4096, 4097, 4096 + 30, 4096 + 31, 4096 + 50, 8192 + 20, 12288):
        seq = random_dna(n, n)
        for k in (21, 31, 51, 7):
            g, o = pair(0, k, MAX_HASH_1000 * 200, True)
            g.add_sequence(seq); o.add_sequence(seq)
            same(g, o)


# ------------------------------------------------------------------------------------------------
# protein sketches: 6-frame translation (lib.rs:275-302), SURVEY 8(f) rank 4
# ------------------------------------------------------------------------------------------------
def ppair(num, k, max_hash=0, abund=False):
    return smb.KmerMinHash(num, k, True, 42, max_hash, abund), orc.KmerMinHash(num, k, True, 42, max_hash, abund)


@pytest.mark.parametrize("k", [21, 30, 57, 3, 4, 10])
@pytest.mark.parametrize("kind", ["num", "scaled_abund", "num_abund"])
def test_protein_add_sequence_parity(k, kind):
    seq = dirty(random_dna(30011, 0x700 + k), 5 + k, n_bad=40)
    num = 300 if kind.startswith("num") else 0
    mx = 0 if kind.startswith("num") else MAX_HASH_1000 * 100
    g, o = ppair(num, k, mx, kind.endswith("abund"))
    g.add_sequence(seq, False); o.add_sequence(seq, False)  # no validity check in the protein arm
    same(g, o)
    g.add_sequence(seq[:5000], True); o.add_sequence(seq[:5000], True)
    same(g, o)
    for short in (b"", b"AC", b"ACG", b"ACGTACGTAC"[: k - 1], b"ACGTNNACGTACGATCGATCGACTGACTAGCTAGCTAGCATCGAT"):
        g.add_sequence(short, True); o.add_sequence(short, True)
    same(g, o)


def test_protein_batches_and_mixed_sketches():
    genome = random_dna(50_000, 0x5EED0010)
    n_reads = 900
    reads = make_reads(genome, n_reads, 150, 0x5EED0011)
    gp, op = ppair(0, 21, MAX_HASH_1000 * 50, True)
    gd, od = pair(0, 21, MAX_HASH_1000 * 50, True)
    smb.add_reads([gd, gp], reads, n_reads, 150)  # a DNA and a protein sketch from the same pass
    od.add_reads(reads, n_reads, 150); op.add_reads(reads, n_reads, 150)
    same(gp, op); same(gd, od)
    lens = [0, 2, 20, 21, 22, 23, 24, 300, 7, 1000, 0, 64]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    buf = dirty(random_dna(int(offsets[-1]), 3), 4, n_bad=5)
    g, o = ppair(50, 21, 0, True)
    g.add_sequences(buf, offsets)
    for i in range(len(lens)):
        o.add_sequence(buf[int(offsets[i]):int(offsets[i + 1])], True)
    same(g, o)
    with pytest.raises(smb.SourmashError) as e:  # ksize < 3: the reference panics in slice::windows(0)
        smb.KmerMinHash(10, 2, True).add_sequence(b"ACGTACGT")
    assert e.value.code == 1
    # protein and DNA sketches do not compare (lib.rs:179-181)
    with pytest.raises(smb.SourmashError) as e:
        gp.compare(gd)
    assert e.value.code == 102


# ------------------------------------------------------------------------------------------------
# batches: reads and ragged sequences, several sketches per pass
# ------------------------------------------------------------------------------------------------
def test_add_reads_multi_k():  # BASELINE config 2 shape, reduced
    genome = random_dna(200_000, 0x5EED0010)
    n_reads = 20000
    reads = make_reads(genome, n_reads, 150, 0x5EED0011)
    ks = (21, 31, 51)
    gs = [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000, True) for k in ks]
    smb.add_reads(gs, reads, n_reads, 150, force=False)
    os_ = orc.mt_sketch_reads(reads, n_reads, 150, list(ks), 0, MAX_HASH_1000, True, 4)
    for g, o in zip(gs, os_):
        same(g, o)
        assert g.md5sum() == o.md5sum()
    # a second batch accumulates
    reads2 = make_reads(genome, 5000, 150, 0x5EED0012)
    smb.add_reads(gs, reads2, 5000, 150)
    for g, o in zip(gs, os_):
        o.add_reads(reads2, 5000, 150)
        same(g, o)


@pytest.mark.parametrize("ks", [(21, 31), (21, 51), (31, 51), (21, 31, 51), (51, 31, 21), (31, 31, 21), (21, 9, 51, 33)])
def test_fused_multi_k_launch(ks):
    """Batch calls share one fused launch among distinct k in {21, 31, 51} (smgpu_fuse_multi_k): the
    fused kernel, the per-sketch kernels and the oracle must agree -- dirty, ragged input, mixed sketch
    kinds, force on and off (the first failing k-mer differs per k)."""
    r = splitmix64(777 + sum(ks), 200)
    lens = [int(x % np.uint64(900)) for x in r[:150]] + [0, 20, 21, 22, 30, 31, 32, 50, 51, 52, 9000, 0]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    clean = random_dna(int(offsets[-1]), 5 + len(ks))
    buf = dirty(clean, 99)
    kinds = [(0, MAX_HASH_1000 * 40, True), (300, 0, False), (0, MAX_HASH_1000 * 40, False), (150, 0, True)]

    def sketches():
        gs, os_ = [], []
        for j, k in enumerate(ks):
            num, mx, ab = kinds[j % len(kinds)]
            g, o = pair(num, k, mx, ab)
            gs.append(g); os_.append(o)
        return gs, os_

    results = {}
    for fuse in (True, False):
        smb.fuse_multi_k(fuse)
        try:
            gs, os_ = sketches()
            smb.add_sequences(gs, buf, offsets, force=True)
            for o in os_:
                for s in range(len(lens)):
                    o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], True)
            for g, o in zip(gs, os_):
                same(g, o)
            # a second, clean batch of fixed-length reads accumulates into the same sketches
            reads = make_reads(clean[:60000], 700, 150, 31)
            smb.add_reads(gs, reads, 700, 150, force=False)
            for g, o in zip(gs, os_):
                o.add_reads(reads, 700, 150)
                same(g, o)
            results[fuse] = [g.md5sum() for g in gs]
            # force=False on the dirty batch: error of the first sketch that fails, partial state kept
            gs, os_ = sketches()
            with pytest.raises(smb.SourmashError) as ge:
                smb.add_sequences(gs, buf, offsets, force=False)
            msgs = []
            for o in os_:
                msg = None
                for s in range(len(lens)):
                    try:
                        o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], False)
                    except orc.SourmashError as e:
                        msg = e.message
                        break
                msgs.append(msg)
            assert ge.value.message in msgs
            for g, o in zip(gs, os_):
                same(g, o)
        finally:
            smb.fuse_multi_k(True)
    assert results[True] == results[False]


@pytest.mark.parametrize("read_len", [30, 31, 32, 100, 151, 2048, 5000])
def test_add_reads_lengths(read_len):
    n_reads = max(3, 200000 // read_len)
    buf = dirty(random_dna(n_reads * read_len, read_len), read_len, lower=False)
    for k, num, mx in ((31, 0, MAX_HASH_1000 * 50), (21, 200, 0)):
        g, o = pair(num, k, mx, True)
        g.add_reads(buf, n_reads, read_len, force=True)
        o.add_reads(buf, n_reads, read_len, True)
        same(g, o)


def test_add_sequences_ragged():
    r = splitmix64(4242, 400)
    lens = [int(x % np.uint64(700)) for x in r[:300]] + [0, 0, 5000, 1, 20, 21, 22, 0]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    buf = dirty(random_dna(int(offsets[-1]), 11), 12)
    for k, num, mx, ab in ((21, 0, MAX_HASH_1000 * 50, True), (31, 100, 0, False), (9, 64, 0, True)):
        g, o = pair(num, k, mx, ab)
        g.add_sequences(buf, offsets, force=True)
        for s in range(len(lens)):
            o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], True)
        same(g, o)
    # force=False: stops at the first failing k-mer in batch order
    g, o = pair(0, 21, MAX_HASH_1000 * 50, True)
    with pytest.raises(smb.SourmashError) as ge:
        g.add_sequences(buf, offsets, force=False)
    msg = None
    for s in range(len(lens)):
        try:
            o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], False)
        except orc.SourmashError as e:
            msg = e.message
            break
    assert ge.value.message == msg
    same(g, o)


def test_device_resident_input():
    import torch
    genome = random_dna(300_000, 31337)
    t = torch.frombuffer(bytearray(genome), dtype=torch.uint8).cuda()
    g, o = pair(0, 31, MAX_HASH_1000 * 10, True)
    g.add_reads(t.data_ptr(), 1, len(genome), on_device=True)
    o.add_sequence(genome)
    same(g, o)
    out = torch.zeros(g.size(), dtype=torch.int64, device="cuda")
    smb._call("kmerminhash_copy_mins", g._p, smb._vp(out.data_ptr()), None, True)
    assert np.array_equal(out.cpu().numpy().view(np.uint64), o.mins_np())


# ------------------------------------------------------------------------------------------------
# add_hash state machine, merge, pair operations
# ------------------------------------------------------------------------------------------------
def test_add_hash_quirks():
    g, o = pair(3, 21, 0, True)
    for h in (9, 9, 5, 9, 7, 9, 9):  # lib.rs:206-208
        g.add_hash(h); o.add_hash(h)
    same(g, o)
    assert g.mins == [5, 7, 9] and g.abunds == [1, 1, 3]
    g, o = pair(0, 21)  # num=0, max_hash=0: order dependent, replayed
    for h in (50, 100, 20, 70, 10):
        g.add_hash(h); o.add_hash(h)
    same(g, o)
    assert g.mins == [10, 20, 50]
    g, o = pair(0, 21, 100, True)
    for h in (100, 101, 7, 100, 0):
        g.add_hash(h); o.add_hash(h)
    same(g, o)
    g, o = pair(4, 21, 1000, True)  # both set: scaled gate, then truncation
    for h in (900, 5, 1001, 17, 17, 800, 3, 900, 1000, 2):
        g.add_hash(h); o.add_hash(h)
    same(g, o)


@pytest.mark.parametrize("abund", [False, True])
def test_add_hash_random_streams(abund):
    r = splitmix64(2024, 6000) % np.uint64(1500)
    for num, mx in ((50, 0), (0, 700), (20, 900), (0, 0)):
        g, o = pair(num, 21, mx, abund)
        # interleave reads of the state with the stream (flush points)
        for chunk in np.array_split(r, 7):
            g.add_many(chunk.tolist() if len(chunk) < 50 else chunk[:50].tolist())
            o.add_many(chunk[:50])
            same(g, o)
        lib = smb.lib()
        rest = np.ascontiguousarray(r[:3000])
        for h in rest.tolist():
            lib.kmerminhash_add_hash(g._p, h)
        o.add_many(rest)
        same(g, o)


@pytest.mark.parametrize("abund", [False, True])
def test_scaled_fold_paths(abund):
    """Folding candidates into a scaled sketch that already holds hashes: candidates found in the state only
    bump abundances; new ones are merged in by the one-CTA sort (up to 2048 of them) or by the generic union.
    Batches are sized to land on every path and on the boundaries, with repeats inside a batch."""
    mx = MAX_HASH_1000 * 100
    pool = splitmix64(31 + abund, 40000) % np.uint64(mx)
    g, o = pair(0, 31, mx, abund)
    cursor = 0
    for n_new in (3000, 0, 1, 7, 2047, 2048, 2049, 5000, 0, 300):
        fresh = pool[cursor:cursor + n_new]
        cursor += n_new
        seen = pool[:cursor - n_new]
        old = seen[:: max(1, len(seen) // 900)] if len(seen) else seen  # hashes the sketch already holds
        batch = np.concatenate([fresh, old, fresh[::3], old[::2], np.array([mx + 5, mx + 1], dtype=np.uint64)])
        rng = splitmix64(cursor + 1, len(batch))
        batch = batch[np.argsort(rng, kind="stable")]  # shuffled
        g.add_many(batch)
        o.add_many(batch)
        same(g, o)  # reading the sketch folds the candidates
    assert g.md5sum() == o.md5sum()


def test_add_word_and_add_from():
    g, o = pair(10, 5)
    for w in (b"ACGTA", b"hello", b"x" * 40, b"ACG"):
        g.add_word(w); o.add_word(w)
    same(g, o)
    g2, o2 = pair(3, 5)
    g2.add_from(g); o2.add_from(o)
    same(g2, o2)


@pytest.mark.parametrize("ta,tb", [(False, False), (True, True), (True, False), (False, True)])
@pytest.mark.parametrize("num,mx", [(40, 0), (0, MAX_HASH_1000 * 300), (1000, 0)])
def test_merge_parity(ta, tb, num, mx):
    s1, s2 = random_dna(5000, 1), random_dna(5000, 2)
    ga, oa = pair(num, 21, mx, ta)
    gb, ob = pair(num, 21, mx, tb)
    for s in (s1, s1[:2000]):
        ga.add_sequence(s); oa.add_sequence(s)
    for s in (s2, s1[1000:3000]):
        gb.add_sequence(s); ob.add_sequence(s)
    ga.merge(gb); oa.merge(ob)
    assert ga.track_abundance() == oa.track_abundance()
    same(ga, oa)
    same(gb, ob)


def test_check_compatible_order():  # lib.rs:176-190
    a = smb.KmerMinHash(10, 21)
    for args, code in (((10, 31), 101), ((10, 21, True), 102), ((10, 21, False, 42, 5), 103),
                       ((10, 21, False, 43), 104)):
        for op in (a.compare, a.count_common, a.merge):
            with pytest.raises(smb.SourmashError) as e:
                op(smb.KmerMinHash(*args))
            assert e.value.code == code
        assert a.intersection_union_size(smb.KmerMinHash(*args)) == 0  # ffi.rs:304-307: swallowed


def test_pair_ops_random():
    base = random_dna(30000, 8)
    for num, mx in ((500, 0), (0, MAX_HASH_1000 * 30), (64, 0)):
        sk = []
        for i, rate in enumerate((0.0, 0.002, 0.02, 0.2)):
            g, o = pair(num, 21, mx)
            s = mutate(base, rate, 100 + i)[: 30000 - 3000 * i]
            g.add_sequence(s); o.add_sequence(s)
            sk.append((g, o))
        empty = pair(num, 21, mx)
        sk.append(empty)
        for ga, oa in sk:
            for gb, ob in sk:
                assert ga.count_common(gb) == oa.count_common(ob)
                assert ga.compare(gb) == oa.compare(ob)
                c = ga.containment(gb)
                oc = oa.containment(ob)
                assert (np.isnan(c) and np.isnan(oc)) or c == oc


# ------------------------------------------------------------------------------------------------
# collections: all-vs-all matrix and linear search
# ------------------------------------------------------------------------------------------------
def _planted_rows(n_rows, n_hashes, seed, max_hash=None):
    """sorted-unique u64 rows with planted shared subsets (SURVEY 8(d) cfg3 compare-only input)"""
    rows = []
    pool = splitmix64(seed, n_hashes * 4)
    if max_hash:
        pool = pool % np.uint64(max_hash)
    for i in range(n_rows):
        own = splitmix64(seed + 1000 + i, n_hashes)
        if max_hash:
            own = own % np.uint64(max_hash)
        frac = (i % 7) / 8.0
        take = int(n_hashes * frac)
        start = (i * 37) % (len(pool) - take + 1)
        r = np.unique(np.concatenate([own[: n_hashes - take], pool[start:start + take]]))
        rows.append(r)
    return rows


@pytest.fixture
def compare_path(request):
    smb.compare_path(request.param)
    yield request.param
    smb.compare_path("auto")


@contextlib.contextmanager
def scope_counts(*kinds):
    """Launches per profiler scope inside the block (profiling on: one stream): got[kind] afterwards."""
    for kd in kinds:
        smb.profile_read(kd, reset=True)
    got = {}
    smb.profile_enable(True)
    try:
        yield got
    finally:
        smb.profile_enable(False)
        for kd in kinds:
            got[kd] = smb.profile_read(kd, reset=True)[1]


@pytest.mark.parametrize("compare_path", ["auto", "dense", "sparse"], indirect=True)
@pytest.mark.parametrize("num,n_hashes,mx", [(500, 500, 0), (0, 1200, MAX_HASH_1000 * 50), (100, 130, 0)])
def test_compare_matrix_vs_oracle(num, n_hashes, mx, compare_path):
    rows = _planted_rows(96, n_hashes, 17 + num, mx or None)
    if num:
        rows = [r[:num] for r in rows]
    rows[5] = rows[5][:0]  # an empty sketch
    rows[6] = rows[6][:1]
    g_sk, o_sk = [], []
    for r in rows:
        g, o = pair(num, 31, mx)
        g.set_mins(r)
        for v in r:
            o.mins_push(int(v))
        g_sk.append(g); o_sk.append(o)
    coll = smb.SketchCollection.from_sketches(g_sk)
    offsets = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.uint64)
    coll2 = smb.SketchCollection.from_csr(np.concatenate(rows), offsets, len(rows), num, 31, 42, mx)
    oc, osz = orc.compare_matrix(o_sk, o_sk)
    occ = orc.count_common_matrix(o_sk, o_sk)
    for c in (coll, coll2):
        common, size, ratio = smb.compare_matrix(c, c, "compare")
        assert np.array_equal(common, oc) and np.array_equal(size, osz)
        assert np.array_equal(ratio, oc.astype(np.float64) / np.maximum(1, osz).astype(np.float64))
        common, size, ratio = smb.compare_matrix(c, c, "containment")
        assert np.array_equal(common, occ)
        assert np.array_equal(size, np.repeat(np.array([len(r) for r in rows], dtype=np.uint32)[:, None], len(rows), 1))
    # a rectangular sub-block
    common, size, ratio = smb.compare_matrix(coll, coll2, "compare", r0=10, nr=37, c0=3, nc=50)
    assert np.array_equal(common, oc[10:47, 3:53]) and np.array_equal(size, osz[10:47, 3:53])
    # linear search, both modes, several thresholds: hits and their order
    queries = smb.SketchCollection.from_sketches(g_sk[:9])
    for mode in ("similarity", "containment"):
        for thr in (0.0, 0.1, 0.5):
            got = smb.linear_find(coll, queries, mode, thr)
            for q in range(9):
                assert got[q] == orc.linear_find(o_sk, o_sk[q], mode, thr)


@pytest.mark.parametrize("compare_path", ["auto", "sparse", "dense"], indirect=True)
@pytest.mark.parametrize("num,n_hashes,mx", [(400, 400, 0), (0, 900, MAX_HASH_1000 * 50)])
def test_compare_row_shards_and_query_batches(num, n_hashes, mx, compare_path):
    """Row blocks much narrower than the column block -- a rank's shard of the all-vs-all matrix, a query
    batch against an index -- take the probe form of the join (a hash table over the smaller side); every
    path must give the oracle's integers."""
    rows = _planted_rows(240, n_hashes, 91 + num, mx or None)
    if num:
        rows = [r[:num] for r in rows]
    rows[50] = rows[50][:0]
    rows[51] = rows[51][:2]
    for i in range(140, 160):  # a shard of empty sketches only
        rows[i] = rows[i][:0]
    g_sk, o_sk = [], []
    for r in rows:
        g, o = pair(num, 31, mx)
        g.set_mins(r)
        for v in r:
            o.mins_push(int(v))
        g_sk.append(g); o_sk.append(o)
    coll = smb.SketchCollection.from_sketches(g_sk)
    oc, osz = orc.compare_matrix(o_sk, o_sk)
    occ = orc.count_common_matrix(o_sk, o_sk)
    lens = np.array([len(r) for r in rows], dtype=np.uint32)
    for r0, nr in ((0, 30), (40, 60), (200, 40), (50, 2)):  # shards of the same collection
        common, size, ratio = smb.compare_matrix(coll, coll, "compare", r0=r0, nr=nr)
        assert np.array_equal(common, oc[r0:r0 + nr]) and np.array_equal(size, osz[r0:r0 + nr])
        assert np.array_equal(ratio, oc[r0:r0 + nr].astype(np.float64) / np.maximum(1, osz[r0:r0 + nr]).astype(np.float64))
        common, size, ratio = smb.compare_matrix(coll, coll, "containment", r0=r0, nr=nr)
        assert np.array_equal(common, occ[r0:r0 + nr])
        assert np.array_equal(size, np.repeat(lens[r0:r0 + nr, None], len(rows), 1))
    # The shard of empty rows: the probe form builds an empty table and writes every cell as unrelated.  As the
    # first block of its collection it takes the probe form on "auto" too (20 x 240 cells: past the size threshold).
    r0, nr = 140, 20
    assert nr * len(rows) >= 4096
    fresh = smb.SketchCollection.from_sketches(g_sk)
    with scope_counts("compare_probe") as probed:
        common, size, ratio = smb.compare_matrix(fresh, fresh, "compare", r0=r0, nr=nr)
        ccommon, csize, _ = smb.compare_matrix(fresh, fresh, "containment", r0=r0, nr=nr)
    assert np.array_equal(common, oc[r0:r0 + nr]) and np.array_equal(size, osz[r0:r0 + nr])
    assert np.array_equal(ratio, oc[r0:r0 + nr].astype(np.float64) / np.maximum(1, osz[r0:r0 + nr]).astype(np.float64))
    assert np.array_equal(ccommon, occ[r0:r0 + nr]) and not csize.any()
    if compare_path != "dense":
        assert probed["compare_probe"] == 2
    # a separate (small) query collection as the ROW side, the index as columns, and the other way round
    queries = smb.SketchCollection.from_sketches(g_sk[100:120])
    common, size, ratio = smb.compare_matrix(queries, coll, "compare")
    assert np.array_equal(common, oc[100:120]) and np.array_equal(size, osz[100:120])
    common, size, ratio = smb.compare_matrix(queries, coll, "containment")
    assert np.array_equal(common, occ[100:120])
    common, size, ratio = smb.compare_matrix(coll, queries, "containment")
    assert np.array_equal(common, occ[:, 100:120])
    for mode in ("similarity", "containment"):
        got = smb.linear_find(coll, queries, mode, 0.1)
        for q in range(20):
            assert got[q] == orc.linear_find(o_sk, o_sk[100 + q], mode, 0.1)


@pytest.mark.parametrize("compare_path", ["dense", "sparse"], indirect=True)
def test_compare_mostly_unrelated_clusters(compare_path):
    # the shape the sparse path is for: clusters of related sketches, everything else disjoint
    import bench
    N = 600
    rows = bench.planted_sketches(N, 500, 99)
    rows[17] = rows[16]  # identical pair
    offs = np.arange(N + 1, dtype=np.uint64) * np.uint64(500)
    coll = smb.SketchCollection.from_csr(rows.reshape(-1), offs, N, 500, 31)
    common, size, ratio = smb.compare_matrix(coll, coll, "compare")
    ccommon, csize, cratio = smb.compare_matrix(coll, coll, "containment")
    osk = []
    for i in range(N):
        o = orc.KmerMinHash(500, 31)
        o.add_many(rows[i])
        osk.append(o)
    oc, osz = orc.compare_matrix(osk, osk, 4)
    assert np.array_equal(common, oc) and np.array_equal(size, osz)
    assert np.array_equal(ratio, oc / np.maximum(1, osz))
    assert np.array_equal(ccommon[:200, :200], orc.count_common_matrix(osk[:200], osk[:200]))
    assert (csize == 500).all() and np.array_equal(cratio, ccommon / 500.0)
    assert common[16, 17] == 500 and ratio[16, 17] == 1.0
    # row-sharded block of the same collection (the rows are part of the columns) ...
    c2, s2, r2 = smb.compare_matrix(coll, coll, "compare", r0=100, nr=150, c0=0, nc=N)
    assert np.array_equal(c2, oc[100:250]) and np.array_equal(s2, osz[100:250])
    c2, s2, r2 = smb.compare_matrix(coll, coll, "containment", r0=100, nr=150, c0=50, nc=300)
    assert np.array_equal(c2, ccommon[100:250, 50:350])
    # ... and a row range that sticks out of the column range
    c2, s2, r2 = smb.compare_matrix(coll, coll, "compare", r0=0, nr=300, c0=200, nc=300)
    assert np.array_equal(c2, oc[0:300, 200:500]) and np.array_equal(r2, (oc / np.maximum(1, osz))[0:300, 200:500])


@pytest.mark.parametrize("compare_path", ["auto", "dense", "sparse"], indirect=True)
def test_compare_mostly_related_full_sketches(compare_path):
    # one big family: every pair shares most hashes -> the data-driven choice is the dense walk,
    # which for full num sketches runs on 32-bit ranks with a fixed trip count
    r = np.random.Generator(np.random.PCG64(12))
    N, NUM = 150, 256
    root = np.unique(r.integers(0, 1 << 63, size=3 * NUM, dtype=np.uint64))
    rows = np.empty((N, NUM), dtype=np.uint64)
    for i in range(N):
        kept = root[r.random(root.size) < 0.8]
        fresh = r.integers(0, 1 << 63, size=NUM, dtype=np.uint64)
        rows[i] = np.unique(np.concatenate([kept, fresh]))[:NUM]
    rows[3] = rows[2]
    offs = np.arange(N + 1, dtype=np.uint64) * np.uint64(NUM)
    coll = smb.SketchCollection.from_csr(rows.reshape(-1), offs, N, NUM, 31)
    other = smb.SketchCollection.from_csr(rows[40:110].reshape(-1), offs[:71], 70, NUM, 31)
    osk = []
    for i in range(N):
        o = orc.KmerMinHash(NUM, 31)
        o.add_many(rows[i])
        osk.append(o)
    oc, osz = orc.compare_matrix(osk, osk, 4)
    common, size, ratio = smb.compare_matrix(coll, coll, "compare")
    assert np.array_equal(common, oc) and np.array_equal(size, osz) and np.array_equal(ratio, oc / np.maximum(1, osz))
    assert common[2, 3] == NUM and (size == NUM).all()
    # ragged tile edges, a row-sharded block, and two different collections
    c2, s2, r2 = smb.compare_matrix(coll, coll, "compare", r0=33, nr=70, c0=0, nc=N)
    assert np.array_equal(c2, oc[33:103])
    c2, s2, r2 = smb.compare_matrix(coll, other, "compare", r0=5, nr=100, c0=0, nc=70)
    assert np.array_equal(c2, oc[5:105, 40:110]) and np.array_equal(r2, (oc / np.maximum(1, osz))[5:105, 40:110])


@pytest.mark.parametrize("compare_path", ["auto"], indirect=True)
def test_compare_mostly_related_scaled_sketches(compare_path):
    # one big family of scaled sketches of different lengths: the first block over the rows probes and finds the
    # dense walk the better choice; every later block over the same rows goes to the dense kernel directly
    r = np.random.Generator(np.random.PCG64(13))
    N, mx = 150, MAX_HASH_1000 * 50
    root = np.unique(r.integers(0, mx, size=2000, dtype=np.uint64))
    rows = []
    for i in range(N):
        kept = root[r.random(root.size) < (0.5, 0.7, 0.9)[i % 3]]
        rows.append(np.unique(np.concatenate([kept, r.integers(0, mx, size=int(r.integers(10, 600)), dtype=np.uint64)])))
    gs, osk = [], []
    for row in rows:
        g, o = pair(0, 31, mx)
        g.set_mins(row); o.add_many(row)
        gs.append(g); osk.append(o)
    assert len({len(row) for row in rows}) > 1
    coll = smb.SketchCollection.from_sketches(gs)
    oc, osz = orc.compare_matrix(osk, osk, 4)
    with scope_counts("compare_probe") as first:
        common, size, ratio = smb.compare_matrix(coll, coll, "compare")
    assert np.array_equal(common, oc) and np.array_equal(size, osz) and np.array_equal(ratio, oc / np.maximum(1, osz))
    assert first["compare_probe"] == 1
    with scope_counts("compare_probe", "join_sort", "compare") as again:
        common, size, ratio = smb.compare_matrix(coll, coll, "compare")
    assert np.array_equal(common, oc) and np.array_equal(size, osz) and np.array_equal(ratio, oc / np.maximum(1, osz))
    assert again["compare_probe"] == 0 and again["join_sort"] == 0 and again["compare"] >= 1


def test_scaffold_leaf_pairing():  # SURVEY 8(f) rank 2: src/index/sbt.rs:356-381
    g = golden("sbt_v5_leaves.json")
    pos = sorted(g["leaves"], key=int)
    gl = [_load(smb, g["leaves"][p]["sketch"]) for p in pos]
    ol = [_load(orc, g["leaves"][p]["sketch"]) for p in pos]
    got = smb.scaffold_pairs(smb.SketchCollection.from_sketches(gl))
    assert got == orc.scaffold_pairs(ol)
    assert len(got) == 4 and got[-1][1] is None  # 7 leaves -> 3 pairs + 1 single (scaffold_sbt keeps 7 leaves)
    # clusters + unrelated sketches + an odd/even count, scaled sketches of different sizes
    import bench
    rows = bench.planted_sketches(301, 120, 77)
    gs, os_ = [], []
    for i in range(301):
        a, o = pair(120, 31)
        a.set_mins(rows[i]); o.add_many(rows[i])
        gs.append(a); os_.append(o)
    for n in (301, 300, 2, 1):
        assert smb.scaffold_pairs(smb.SketchCollection.from_sketches(gs[:n])) == orc.scaffold_pairs(os_[:n])


def test_unsorted_rows_rejected():  # SURVEY section 4: .sbt.subset fixtures are stored unsorted
    g = golden("subset_scaled.json")
    sk = g["leaves"][0]["sketch"]
    mh = _load(smb, sk)
    assert mh.size() == len(sk["mins"])  # raw pushes are kept as they are
    other = _load(smb, g["leaves"][1]["sketch"])
    with pytest.raises(smb.SourmashError) as e:
        mh.count_common(other)
    assert e.value.code == 2
    with pytest.raises(smb.SourmashError):
        smb.SketchCollection.from_sketches([mh])


def test_cfg4_containment_search_scaled():  # BASELINE config 4 shape, reduced: scaled index, query batch
    r = np.random.Generator(np.random.PCG64(4))
    mx = MAX_HASH_1000 * 4
    index, o_index = [], []
    base = [np.unique(r.integers(0, mx, size=3000, dtype=np.uint64)) for _ in range(12)]
    for i in range(240):
        b = base[i % 12]
        keep = b[r.random(b.size) < (0.1, 0.3, 0.6, 0.9)[i % 4]]
        row = np.unique(np.concatenate([keep, r.integers(0, mx, size=int(r.integers(50, 2500)), dtype=np.uint64)]))
        g, o = pair(0, 31, mx)
        g.set_mins(row); o.add_many(row)
        index.append(g); o_index.append(o)
    queries, o_queries = [], []
    for q in range(10):
        row = np.unique(np.concatenate([base[q][::2], r.integers(0, mx, size=1500, dtype=np.uint64)]))
        g, o = pair(0, 31, mx)
        g.set_mins(row); o.add_many(row)
        queries.append(g); o_queries.append(o)
    ic, qc = smb.SketchCollection.from_sketches(index), smb.SketchCollection.from_sketches(queries)
    for path in ("dense", "sparse", "auto"):
        smb.compare_path(path)
        for mode in ("containment", "similarity"):
            got = smb.linear_find(ic, qc, mode, 0.1)  # threshold of benches/index.rs:33
            for q in range(10):
                assert got[q] == orc.linear_find(o_index, o_queries[q], mode, 0.1), (path, mode, q)
    smb.compare_path("auto")
    assert any(len(h) for h in got)


@pytest.mark.parametrize("k", [21, 31, 51, 9])
@pytest.mark.parametrize("num,mx", [(0, MAX_HASH_1000 * 20), (120, 0)])
def test_sketch_collection_one_pass(k, num, mx):
    """smgpu_sketch_collection: one fresh sketch per sequence in a single pass == the loop of
    new + add_sequence(force=true) + push, for scaled and num sketches, ragged lengths (empty, shorter than k,
    a few much shorter than the median so that the num threshold estimate cuts them short), dirty input."""
    r = splitmix64(5150 + k + num, 64)
    lens = [int(20000 + x % np.uint64(9000)) for x in r[:14]] + [0, k - 1, k, k + 5, 300, 2500, 0, 60000]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    buf = dirty(random_dna(int(offsets[-1]), 77 + k), 88, n_bad=40)
    # two sequences share most of their content (related sketches), one is a repeat of a short motif
    a, b = int(offsets[1]), int(offsets[2])
    buf = buf[:a] + buf[:b - a] + buf[b:]
    m0 = int(offsets[5])
    motif = (b"ACGTTGCA" * 4000)[: lens[5]]
    buf = buf[:m0] + motif + buf[m0 + lens[5]:]
    coll = smb.SketchCollection.sketch_sequences(buf, offsets, num, k, 42, mx)
    assert len(coll) == len(lens)
    rows = coll.rows_np()
    os_ = []
    for s in range(len(lens)):
        o = orc.KmerMinHash(num, k, False, 42, mx, False)
        o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], True)
        os_.append(o)
        assert np.array_equal(rows[s], o.mins_np()), (s, lens[s], len(rows[s]), o.size())
    # ... and the collection behaves like one built by pushing the sketches
    common, size, ratio = smb.compare_matrix(coll, coll, "compare")
    oc, osz = orc.compare_matrix(os_, os_)
    assert np.array_equal(common, oc) and np.array_equal(size, osz)
    # device-resident input gives the same rows
    import torch
    t = torch.frombuffer(bytearray(buf + b"\0" * 64), dtype=torch.uint8).cuda()
    to = torch.from_numpy(offsets.view(np.int64)).cuda()
    coll2 = smb.SketchCollection.sketch_sequences(t.data_ptr(), to.data_ptr(), num, k, 42, mx, on_device=True, n_seqs=len(lens))
    for x, y in zip(rows, coll2.rows_np()):
        assert np.array_equal(x, y)


def test_cfg5_sketch_then_all_vs_all():  # BASELINE config 5 shape, reduced: genomes -> scaled sketches -> matrix
    roots = [random_dna(120_000, 0x5EED2000 + c) for c in range(4)]
    gs, os_ = [], []
    for i in range(24):
        genome = mutate(roots[i % 4], (0.001, 0.005, 0.01, 0.02, 0.05)[i % 5], 7000 + i)
        g, o = pair(0, 31, MAX_HASH_1000 * 10)
        g.add_sequence(genome); o.add_sequence(genome)
        gs.append(g); os_.append(o)
    coll = smb.SketchCollection.from_sketches(gs)
    for path in ("dense", "sparse"):
        smb.compare_path(path)
        common, size, ratio = smb.compare_matrix(coll, coll, "compare")
        oc, osz = orc.compare_matrix(os_, os_)
        assert np.array_equal(common, oc) and np.array_equal(size, osz)
        assert np.array_equal(ratio, oc / np.maximum(1, osz))
    smb.compare_path("auto")
    assert ratio[0, 4] > 0.05 and ratio[0, 1] < 0.01  # same root (0.1% vs 5% mutated) vs different roots


# ------------------------------------------------------------------------------------------------
# Signature JSON
# ------------------------------------------------------------------------------------------------
def test_signature_json_example():  # SURVEY 8(a) worked example
    mh = smb.KmerMinHash(20, 10)
    mh.add_sequence(b"TGCCGCCCAGCA")
    sig = smb.Signature()
    sig.push_mh(mh)
    want = ('{"class":"sourmash_signature","email":"","hash_function":"0.murmur64","filename":null,"name":null,'
            '"license":"CC0","signatures":[{"num":20,"ksize":10,"seed":42,"max_hash":0,"mins":[2996412506971915891,'
            '9390240264282449587,14682565545778736889],"md5sum":"2cf8551b3a1c7201168bfb674470319d","molecule":"DNA"}],'
            '"version":0.4}')
    assert sig.save_json().decode() == want
    assert smb.signatures_save_buffer([sig, sig]).decode() == "[" + want + "," + want + "]"


def test_signature_json_vs_oracle_and_roundtrip():
    seq = random_dna(40000, 3)
    gs, os_ = [], []
    for k, num, mx, ab in ((21, 500, 0, False), (31, 0, MAX_HASH_1000 * 10, True), (51, 10, 0, True)):
        g, o = pair(num, k, mx, ab)
        g.add_sequence(seq); o.add_sequence(seq)
        gs.append(g); os_.append(o)
    sig = smb.Signature()
    sig.set_name('genome "x"\té')
    sig.set_filename("a/b\\c.fa")
    for g in gs:
        sig.push_mh(g)
    js = sig.save_json()
    assert js == orc.signature_json(os_, name='genome "x"\té', filename="a/b\\c.fa")
    parsed = json.loads(js)
    assert [s["ksize"] for s in parsed["signatures"]] == [21, 31, 51]
    # load (one Signature per sketch, filters) and save again
    loaded = smb.signatures_load_buffer(b"[" + js + b"]")
    assert len(loaded) == 3 and loaded[0].name == 'genome "x"\té' and loaded[0].license == "CC0"
    for s, g in zip(loaded, gs):
        m = s.first_mh()
        assert np.array_equal(m.mins_np(), g.mins_np())
    assert len(smb.signatures_load_buffer(b"[" + js + b"]", ksize=31)) == 1
    assert len(smb.signatures_load_buffer(b"[" + js + b"]", select_moltype="DNA")) == 3
    assert len(smb.signatures_load_buffer(b"[" + js + b"]", select_moltype="protein")) == 0
    # scaled sketches come back with num = 0 (lib.rs:124)
    assert loaded[1].first_mh().num == 0
    assert loaded[0] == loaded[0]
    with pytest.raises(smb.SourmashError):
        smb.signatures_load_buffer(b"[{\"signatures\": 3}]")


def test_signature_fixture_file():  # tests/signature.rs:10-32 through the golden copy
    s = golden("genome_s10_s11.json")
    doc = [{"class": s["class"], "email": s["email"], "filename": s["filename"], "name": s["name"],
            "hash_function": s["hash_function"], "license": "CC0", "version": 0.4, "signatures": s["sketches"]}]
    sigs = smb.signatures_load_buffer(json.dumps(doc).encode())
    assert len(sigs) == 4
    assert sigs[0].name == s["name"] and sigs[0].filename == s["filename"]
    assert len(smb.signatures_load_buffer(json.dumps(doc).encode(), ksize=21, select_moltype="dna")) == 1
    for sg, sk in zip(sigs, s["sketches"]):
        assert sg.first_mh().md5sum() == sk["md5sum"]
        assert json.loads(sg.save_json())["signatures"][0]["mins"] == sk["mins"]


def test_collection_from_signatures():  # JSON -> CSR in one call == pushing each first sketch (linear.rs:33-36)
    s = golden("sbt_v5_leaves.json")
    doc = [{"hash_function": "0.murmur64", "name": lf["sig_name"], "filename": lf["filename"], "signatures": [lf["sketch"]]}
           for _, lf in sorted(s["leaves"].items(), key=lambda kv: int(kv[0]))]
    sigs = smb.signatures_load_buffer(json.dumps(doc).encode())
    a = smb.SketchCollection.from_signatures(sigs)
    b = smb.SketchCollection.from_sketches([sg.first_mh() for sg in sigs])
    assert len(a) == len(b) == len(sigs)
    for x, y in zip(a.rows_np(), b.rows_np()):
        assert np.array_equal(x, y)
    ca, sa, ra = smb.compare_matrix(a, a)
    cb, sb_, rb = smb.compare_matrix(b, b)
    assert np.array_equal(ca, cb) and np.array_equal(sa, sb_) and np.array_equal(ra, rb)


# ------------------------------------------------------------------------------------------------
# size-independent properties at BASELINE sizes (no oracle run needed)
# ------------------------------------------------------------------------------------------------
def test_full_size_properties():
    n = 5_000_000  # BASELINE config 1 genome length
    g0 = random_dna(n, 0x5EED0001)
    whole = smb.KmerMinHash(0, 31, False, 42, MAX_HASH_1000, True)
    whole.add_sequence(g0)
    # sharded sketching + merge == sketching the whole (shards overlap by k-1 bases)
    parts = [smb.KmerMinHash(0, 31, False, 42, MAX_HASH_1000, True) for _ in range(4)]
    cuts = [0, 1_234_567, 2_500_000, 4_000_001, n]
    for p, a, b in zip(parts, cuts[:-1], cuts[1:]):
        p.add_sequence(g0[a:min(n, b + 30)])
    acc = parts[0]
    for p in parts[1:]:
        acc.merge(p)
    assert np.array_equal(acc.mins_np(), whole.mins_np())
    assert np.array_equal(acc.abunds_np(), whole.abunds_np())
    assert int(whole.abunds_np().sum()) >= whole.size()
    m = whole.mins_np()
    assert (m[1:] > m[:-1]).all() and m[-1] <= MAX_HASH_1000
    # reverse complement has the same canonical k-mers
    rc = smb.KmerMinHash(0, 31, False, 42, MAX_HASH_1000, True)
    rc.add_sequence(g0.translate(bytes.maketrans(b"ACGT", b"TGCA"))[::-1])
    assert np.array_equal(rc.mins_np(), m) and np.array_equal(rc.abunds_np(), whole.abunds_np())
    # num sketch = the smallest `num` of the scaled sketch's universe; idempotent re-add
    nm = smb.KmerMinHash(500, 31)
    nm.add_sequence(g0)
    assert np.array_equal(nm.mins_np(), m[:500])
    nm.add_sequence(g0)
    assert np.array_equal(nm.mins_np(), m[:500])
    assert nm.compare(nm) == 1.0
    g1 = mutate(g0, 0.01, 0x5EED0002)
    nm1 = smb.KmerMinHash(500, 31)
    nm1.add_sequence(g1)
    j = nm.compare(nm1)
    assert 0.4 < j < 0.75 and j == nm1.compare(nm)  # ~ 0.99^31 / (2 - 0.99^31) = 0.58
