"""CPU tests: pin the oracle (oracle/oracle.c) against every known-answer test
and fixture the reference holds for the sketch-and-compare path (SURVEY 8(c))."""
import json

import numpy as np
import pytest

from oracle import oracle as orc
from util import golden, random_dna, MAX_HASH_1000


def test_murmur_kat():  # tests/test.rs:3-6
    assert orc.hash_murmur(b"ACG", 42) == 1731421407650554201


def test_murmur_smhasher_verification():
    # public SMHasher verification value for MurmurHash3_x64_128; pins the 16-byte
    # body loop that no reference test reaches
    assert orc.lib().orc_smhasher_verification() == 0x6384BA69


def test_murmur_body_vectors():  # restatement-derived regression vectors, SURVEY 8(c)
    assert orc.hash_murmur(b"GTCACCCGGTGCTGGGCGGCA") == 529147935188082428
    assert orc.hash_murmur(b"GCTCAACCTAGTCACCCGGTGCTGGGCGGCA") == 13824550005532878703
    assert orc.hash_murmur(b"CTCATTGCAGGTTAATCATGGCTCAACCTAGTCACCCGGTGCTGGGCGGCA") == 14476355676789784531


def test_throws_error():  # tests/minhash.rs:5-17
    mh = orc.KmerMinHash(1, 4)
    with pytest.raises(orc.SourmashError) as e:
        mh.add_sequence(b"ATGR", False)
    assert e.value.code == 1101
    assert e.value.message == "invalid DNA character in input k-mer: ATGR"


def test_merge_kat():  # tests/minhash.rs:19-52
    a, b = orc.KmerMinHash(20, 10), orc.KmerMinHash(20, 10)
    a.add_sequence(b"TGCCGCCCAGCA"); b.add_sequence(b"TGCCGCCCAGCA")
    a.add_sequence(b"GTCCGCCCAGTGA"); b.add_sequence(b"GTCCGCCCAGTGG")
    a.merge(b)
    assert a.mins == [2996412506971915891, 4448613756639084635, 8373222269469409550, 9390240264282449587,
                      11085758717695534616, 11668188995231815419, 11760449009842383350, 14682565545778736889]
    assert a.abunds == []  # merge forces abunds to Some(..), lib.rs:393


def test_compare():  # tests/minhash.rs:54-83
    s1 = b"TGCCGCCCAGCACCGGGTGACTAGGTTGAGCCATGATTAACCTGCAATGA"
    s2 = b"GATTGGTGCACACTTAACTGGGTGCCGCGCTGGTGCTGATCCATGAAGTT"
    a, b = orc.KmerMinHash(20, 10), orc.KmerMinHash(20, 10)
    a.add_sequence(s1); b.add_sequence(s1)
    assert a.compare(b) == 1.0 and b.compare(a) == 1.0
    b.add_sequence(s1)
    assert a.compare(b) == 1.0 and b.compare(a) == 1.0
    b.add_sequence(s2)
    assert a.compare(b) >= 0.3 and b.compare(a) >= 0.3


def _load(sk):
    mh = orc.KmerMinHash(0 if sk["max_hash"] else sk["num"], sk["ksize"], sk["molecule"] == "protein",
                         sk["seed"], sk["max_hash"], "abundances" in sk)
    for m in sk["mins"]:
        mh.mins_push(m)
    for a in sk.get("abundances", []):
        mh.abunds_push(a)
    return mh


def test_sbt_v5_linear_find():  # src/index/sbt.rs:543-588
    g = golden("sbt_v5_leaves.json")
    pos = sorted(g["leaves"], key=int)
    leaves = [_load(g["leaves"][p]["sketch"]) for p in pos]
    q = leaves[pos.index(g["query_position"])]
    want = g["asserted_hits"]
    assert len(orc.linear_find(leaves, q, "similarity", 0.5)) == want["similarity@0.5"]
    assert len(orc.linear_find(leaves, q, "similarity", 0.1)) == want["similarity@0.1"]
    assert len(orc.linear_find(leaves, q, "containment", 0.5)) == want["containment@0.5"]
    assert len(orc.linear_find(leaves, q, "containment", 0.1)) == want["containment@0.1"]
    # the hits themselves (tree positions), SURVEY 8(c)
    assert [int(pos[i]) for i in orc.linear_find(leaves, q, "similarity", 0.1)] == [7, 11]
    assert [int(pos[i]) for i in orc.linear_find(leaves, q, "containment", 0.1)] == [6, 7, 9, 11]


V5_COMPARE = [[500, 43, 0, 37, 0, 39, 0], [43, 500, 0, 39, 0, 178, 0], [0, 0, 500, 0, 191, 0, 182],
              [37, 39, 0, 500, 0, 36, 0], [0, 0, 191, 0, 500, 0, 193], [39, 178, 0, 36, 0, 500, 0],
              [0, 0, 182, 0, 193, 0, 500]]
V5_COMMON = [[500, 54, 0, 61, 0, 55, 0], [54, 500, 0, 70, 0, 268, 0], [0, 0, 500, 0, 267, 0, 275],
             [61, 70, 0, 500, 0, 68, 0], [0, 0, 267, 0, 500, 0, 273], [55, 268, 0, 68, 0, 500, 0],
             [0, 0, 275, 0, 273, 0, 500]]


def test_sbt_v5_matrices():  # SURVEY 8(c) golden integers
    g = golden("sbt_v5_leaves.json")
    leaves = [_load(g["leaves"][p]["sketch"]) for p in sorted(g["leaves"], key=int)]
    common, size = orc.compare_matrix(leaves, leaves)
    assert common.tolist() == V5_COMPARE
    assert (size == 500).all()
    assert orc.count_common_matrix(leaves, leaves).tolist() == V5_COMMON


def test_sbt_v5_intersection_hashes():  # lib.rs:438-468 over the same fixture: as many hashes as `compare` counts
    g = golden("sbt_v5_leaves.json")
    leaves = [_load(g["leaves"][p]["sketch"]) for p in sorted(g["leaves"], key=int)]
    for i in range(7):
        for j in range(7):
            hashes, size = leaves[i].intersection(leaves[j])
            assert (len(hashes), size) == (V5_COMPARE[i][j], 500)
            a, b = set(leaves[i].mins_np().tolist()), set(leaves[j].mins_np().tolist())
            union_bottom = set(sorted(a | b)[:500])
            assert hashes.tolist() == sorted(a & b & union_bottom)


def test_md5sum_fixtures():  # lib.rs:72-77 rule reproduces the stored md5sum of all sorted fixtures
    g = golden("sbt_v5_leaves.json")
    for leaf in g["leaves"].values():
        assert _load(leaf["sketch"]).md5sum() == leaf["sketch"]["md5sum"] == leaf["filename"]
    s = golden("genome_s10_s11.json")
    assert s["n_signatures"] == 1 and len(s["sketches"]) == 4  # tests/signature.rs
    for sk in s["sketches"]:
        assert _load(sk).md5sum() == sk["md5sum"]


def test_md5_rfc1321():
    assert orc.md5_hex(b"") == "d41d8cd98f00b204e9800998ecf8427e"
    assert orc.md5_hex(b"message digest") == "f96b697d7cb7938d525a2f31aaf161d0"
    assert orc.md5_hex(b"1234567890" * 8) == "57edf4a22be3c955ac49da2e2107b67a"


def test_signature_json_example():  # SURVEY 8(a) worked example
    mh = orc.KmerMinHash(20, 10)
    mh.add_sequence(b"TGCCGCCCAGCA")
    want = ('{"class":"sourmash_signature","email":"","hash_function":"0.murmur64","filename":null,"name":null,'
            '"license":"CC0","signatures":[{"num":20,"ksize":10,"seed":42,"max_hash":0,"mins":[2996412506971915891,'
            '9390240264282449587,14682565545778736889],"md5sum":"2cf8551b3a1c7201168bfb674470319d","molecule":"DNA"}],'
            '"version":0.4}')
    assert orc.signature_json([mh]).decode() == want
    json.loads(want)


def test_add_hash_state_machine_quirks():
    # SURVEY 7: full-sketch-max abundance quirk (lib.rs:206-208)
    mh = orc.KmerMinHash(3, 21, track_abundance=True)
    for h in (9, 9, 5, 9, 7, 9, 9):
        mh.add_hash(h)
    assert mh.mins == [5, 7, 9] and mh.abunds == [1, 1, 3]
    # degenerate num=0,max_hash=0: keeps first hash and anything smaller
    mh = orc.KmerMinHash(0, 21)
    for h in (50, 100, 20, 70, 10):
        mh.add_hash(h)
    assert mh.mins == [10, 20, 50]
    # scaled: inclusive max_hash
    mh = orc.KmerMinHash(0, 21, max_hash=100, track_abundance=True)
    for h in (100, 101, 7, 100, 0):
        mh.add_hash(h)
    assert mh.mins == [0, 7, 100] and mh.abunds == [1, 1, 2]


def test_short_and_forced_sequences():
    mh = orc.KmerMinHash(10, 5)
    mh.add_sequence(b"ACG")  # shorter than k: silently ok (lib.rs:257)
    assert mh.size() == 0
    with pytest.raises(orc.SourmashError):
        mh.add_sequence(b"ACNNN")  # len == k, one window, invalid
    assert mh.size() == 0
    mh2 = orc.KmerMinHash(10, 3)
    mh2.add_sequence(b"ACGNACG", True)  # force skips windows overlapping N
    ref = orc.KmerMinHash(10, 3)
    ref.add_sequence(b"ACG")
    assert mh2.mins == ref.mins
    # partial mutation before the error (lib.rs:260-273)
    mh3 = orc.KmerMinHash(10, 3)
    with pytest.raises(orc.SourmashError):
        mh3.add_sequence(b"ACGTNAC", False)
    two = orc.KmerMinHash(10, 3)
    two.add_sequence(b"ACGT")
    assert mh3.mins == two.mins
    # lowercase is uppercased first (lib.rs:253-256)
    lo, up = orc.KmerMinHash(10, 4), orc.KmerMinHash(10, 4)
    lo.add_sequence(b"acgtacgtta"); up.add_sequence(b"ACGTACGTTA")
    assert lo.mins == up.mins


def test_scaled_matches_set_semantics():
    seq = random_dna(20000, 0x5EED0001)
    mh = orc.KmerMinHash(0, 21, max_hash=MAX_HASH_1000 * 50, track_abundance=True)
    mh.add_sequence(seq + seq[:5000])
    from collections import Counter
    cnt = Counter()
    s = seq + seq[:5000]
    tr = bytes.maketrans(b"ACGT", b"TGCA")
    for i in range(len(s) - 20):
        kmer = s[i:i + 21]
        rc = kmer.translate(tr)[::-1]
        h = orc.hash_murmur(min(kmer, rc))
        if h <= MAX_HASH_1000 * 50:
            cnt[h] += 1
    assert mh.mins == sorted(cnt)
    assert mh.abunds == [cnt[h] for h in sorted(cnt)]


@pytest.mark.parametrize("num, k, prot, mx, abund", [
    (0, 21, False, MAX_HASH_1000 * 50, True), (40, 31, False, 0, False), (0, 30, True, 2**64 - 1, False),
    (25, 24, True, 0, True)])
def test_sketch_each_equals_the_per_sequence_loop(num, k, prot, mx, abund):
    lens = [0, 5, 20, 21, 30, 31, 900, 4000, 77, 0, 2500]
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    a = bytearray(random_dna(int(offsets[-1]), 0x5EED0002))
    for p in range(3, len(a), 97):   # invalid bytes and lower case: skipped / upper-cased as add_sequence does
        a[p] = b"Nn-a"[p % 4]
    buf = bytes(a)
    for nthreads in (1, 3, 64):
        got = orc.sketch_each(buf, offsets, num, k, prot, 7, mx, abund, nthreads)
        assert len(got) == len(lens)
        for s, g in enumerate(got):
            o = orc.KmerMinHash(num, k, prot, 7, mx, abund)
            o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], True)
            assert g.mins == o.mins and g.abunds == o.abunds, (nthreads, s)
    assert orc.sketch_each(b"", [0], num, k, prot) == []


def test_check_compatible_order():  # lib.rs:176-190
    a = orc.KmerMinHash(10, 21)
    for args, code in (((10, 31), 101), ((10, 21, True), 102), ((10, 21, False, 42, 5), 103),
                       ((10, 21, False, 43), 104)):
        with pytest.raises(orc.SourmashError) as e:
            a.compare(orc.KmerMinHash(*args))
        assert e.value.code == code


def test_scaffold_leaf_pairing():  # src/index/sbt.rs:356-381 over the v5 fixture (scaffold_sbt test, sbt.rs:592-601)
    g = golden("sbt_v5_leaves.json")
    pos = sorted(g["leaves"], key=int)
    leaves = [_load(g["leaves"][p]["sketch"]) for p in pos]
    pairs = orc.scaffold_pairs(leaves)
    # every leaf appears exactly once: the reference's scaffold keeps all 7 leaves
    seen = sorted([a for a, b in pairs] + [b for a, b in pairs if b is not None])
    assert seen == list(range(7)) and len(pairs) == 4
    # leaf 12 (last) is popped first and pairs with its nearest neighbour by count_common: leaf 8 (275 > 273)
    assert [int(pos[a]) for a, b in pairs][0] == 12 and int(pos[pairs[0][1]]) == 8


# ------------------------------------------------------------------------------------------------
# Nodegraph / SBT (SURVEY 8(f) rank 3): src/index/nodegraph.rs tests and the sbt.find half of load_sbt
# ------------------------------------------------------------------------------------------------
def _oracle_tree():
    from util import sbt_v5_tree
    d, nodes, leaf_positions, t = sbt_v5_tree()
    ngs = {p: (orc.Nodegraph.from_buffer(raw), mnb) for p, (raw, mnb) in nodes.items()}
    leaves = {int(p): _load(v["sketch"]) for p, v in golden("sbt_v5_leaves.json")["leaves"].items()}
    assert sorted(leaves) == leaf_positions
    return d, nodes, ngs, leaves, t


def test_nodegraph_count_and_get():  # nodegraph.rs:236-254
    ng = orc.Nodegraph([10], 3)
    assert ng.count(801084876663808) is True
    assert ng.get(801084876663808) == 1 and ng.unique_kmers() == 1
    assert ng.count(801084876663808) is False and ng.unique_kmers() == 1
    for h in (0, 1, 9, 10, 2**64 - 1, 0x123456789ABCDEF):  # the proptest property on a few values
        g = orc.Nodegraph([10], 3)
        g.count(h)
        assert g.get(h) == 1


def test_nodegraph_load_save_roundtrip():  # nodegraph.rs:256-279: byte-identical re-serialisation
    d, nodes, ngs, leaves, t = _oracle_tree()
    for p, (raw, _) in nodes.items():
        assert ngs[p][0].save() == raw


def test_nodegraph_load_fixture():  # nodegraph.rs:292-821
    d, nodes, ngs, leaves, t = _oracle_tree()
    spec = t["load_nodegraph"]
    ng = ngs[0][0]
    assert ng.tablesizes() == spec["tablesizes"]
    for h in spec["absent"]:
        assert ng.get(h) == 0
    assert len(spec["present"]) == 500
    for h in spec["present"]:
        assert ng.get(h) == 1


def test_nodegraph_update_fixture():  # nodegraph.rs:271-290: internal.1 | internal.2 == internal.0
    d, nodes, ngs, leaves, t = _oracle_tree()
    ng0 = orc.Nodegraph([99991, 99989, 99971, 99961], 1)
    ng0.update(ngs[1][0])
    ng0.update(ngs[2][0])
    assert ng0.save()[19:] == nodes[0][0][19:]  # the bitsets (the header holds ksize / occupied_bins)
    assert ng0.similarity(ngs[0][0]) == 1.0


def test_sbt_find_fixture():  # sbt.rs:543-551: 1 hit above 0.5, 2 above 0.1 for leaf 7
    d, nodes, ngs, leaves, t = _oracle_tree()
    q = leaves[t["asserted_sbt_find"]["query_position"]]
    h5 = orc.sbt_find(d, ngs, leaves, q, "similarity", 0.5)
    h1 = orc.sbt_find(d, ngs, leaves, q, "similarity", 0.1)
    assert len(h5) == t["asserted_sbt_find"]["similarity@0.5"] and len(h1) == t["asserted_sbt_find"]["similarity@0.1"]
    assert h5 == [7] and sorted(h1) == [7, 11]
    # the tree search and the linear scan agree on this fixture (sbt.rs:566-574 asserts the same counts)
    order = sorted(leaves)
    lin = orc.linear_find([leaves[p] for p in order], q, "similarity", 0.1)
    assert sorted(order[i] for i in lin) == sorted(h1)
    # every internal node of the fixture holds all hashes of the leaves below it
    for p, (ng, mnb) in ngs.items():
        below = [l for l in leaves if any(_is_ancestor(p, l, d))]
        for l in below:
            assert ng.matches(leaves[l]) == leaves[l].size()


def _is_ancestor(a, pos, d):
    while pos:
        pos = (pos - 1) // d
        yield pos == a


@pytest.mark.parametrize("tablesizes", [[10], [1, 2, 31, 32, 33], [997, 1009, 1013, 1019], []])
def test_nodegraph_batch_calls_equal_the_per_hash_loop(tablesizes):
    from util import splitmix64
    r = splitmix64(len(tablesizes) + 17, 3000)
    batch = np.concatenate([r, r[::7], np.array([0, 1, 2**63, 2**64 - 1], dtype=np.uint64)])
    one, many = orc.Nodegraph(tablesizes, 21), orc.Nodegraph(tablesizes, 21)
    for part in (batch[:1], batch[1:2000], batch[2000:]):  # the later parts repeat hashes of the earlier ones
        want = [one.count(int(h)) for h in part]
        n, flags = many.count_many(part)
        assert flags.tolist() == want and n == sum(want)
        assert many.save() == one.save() and many.unique_kmers() == one.unique_kmers()
    probe = np.concatenate([r[:500], splitmix64(99, 500)])
    want = [one.get(int(h)) for h in probe]
    n, flags = many.get_many(probe)
    assert flags.tolist() == want and n == sum(want)
    n, flags = many.count_many([])
    assert n == 0 and flags.size == 0


def _walk_by_scan(d, npos, nodes, mnb, lpos, leaves, query, mode, thr):
    """SBT::find with each position looked up by a scan that stops at the first entry (the oracle's earlier form)."""
    hits, stack = [], [0]
    while stack:
        pos = stack.pop()
        if pos in npos:
            i = npos.index(pos)
            v = orc.node_containment(nodes[i], query) if mode == "containment" else orc.node_similarity(nodes[i], mnb[i], query)
            if v > thr:
                stack.extend(d * pos + c + 1 for c in range(d))
        elif pos in lpos:
            i = lpos.index(pos)
            v = leaves[i].containment(query) if mode == "containment" else leaves[i].similarity(query)
            if v > thr:
                hits.append(pos)
    return hits


def _random_tree(d, n_leaves, seed):
    """A heap-layout tree whose internal nodes hold the hashes of the leaves below them, listed in shuffled order."""
    from util import splitmix64
    pool = splitmix64(seed, 4000)
    n_internal = 1
    while n_internal * (d - 1) + 1 < n_leaves:
        n_internal += 1
    lpos = list(range(n_internal, n_internal + n_leaves))
    leaves = []
    for j in range(n_leaves):
        mh = orc.KmerMinHash(0, 31, False, 42, 2**63)
        mh.add_many(np.concatenate([pool[j * 40:j * 40 + 40], pool[3000 + (j // 3) * 50:3000 + (j // 3) * 50 + 50]]) >> np.uint64(1))
        leaves.append(mh)
    npos, nodes, mnb = [], [], []
    for p in range(n_internal):
        below = [leaves[i] for i, lp in enumerate(lpos) if any(_is_ancestor(p, lp, d))]
        ng = orc.Nodegraph([1999, 2003], 31)
        for mh in below:
            ng.count_many(mh.mins_np())
        npos.append(p)
        nodes.append(ng)
        mnb.append(min([mh.size() for mh in below] or [1]))
    order = np.argsort(splitmix64(seed + 1, n_internal))
    return ([npos[i] for i in order], [nodes[i] for i in order], [mnb[i] for i in order]), (lpos, leaves)


def test_sbt_lookup_matches_a_scan():
    """The binary-search position lookup gives the hits the first-match scan gives: on the v5 fixture, on random
    trees, and with a position listed twice (the first entry wins)."""
    d, nodes, ngs, leaves_d, t = _oracle_tree()
    npos, lpos = sorted(ngs), sorted(leaves_d)
    cases = [(d, (npos, [ngs[p][0] for p in npos], [ngs[p][1] for p in npos]), (lpos, [leaves_d[p] for p in lpos]))]
    for dd, nl, seed in ((2, 13, 1), (3, 20, 2), (5, 31, 3)):
        cases.append((dd,) + _random_tree(dd, nl, seed))
    # duplicates: the root listed again after a copy that rejects everything, and a leaf listed twice with different sketches
    dd, (np_, ng_, mb_), (lp_, lv_) = cases[1]
    empty = orc.Nodegraph([1999, 2003], 31)
    cases.append((dd, (np_ + [0], ng_ + [empty], mb_ + [1]), (lp_ + [lp_[0]], lv_ + [lv_[-1]])))
    cases.append((dd, ([0] + np_, [empty] + ng_, [1] + mb_), ([lp_[0]] + lp_, [lv_[-1]] + lv_)))
    n_hits = 0
    for dd, (np_, ng_, mb_), (lp_, lv_) in cases:
        tree = orc.SbtOracle(dd, np_, ng_, mb_, lp_, lv_)
        for q in lv_[:6] + [orc.KmerMinHash(0, 31, False, 42, 2**63)]:
            for mode in ("similarity", "containment"):
                for thr in (0.0, 0.1, 0.5):
                    got = tree.find(q, mode, thr)
                    assert got == _walk_by_scan(dd, np_, ng_, mb_, lp_, lv_, q, mode, thr), (dd, mode, thr)
                    n_hits += len(got)
    assert n_hits > 100
    # the first entry of a duplicated position wins: an empty copy of the root listed first prunes every walk
    dd, (np_, ng_, mb_), (lp_, lv_) = cases[-1]
    assert orc.SbtOracle(dd, np_, ng_, mb_, lp_, lv_).find(lv_[1], "containment", 0.0) == []
    assert orc.SbtOracle(dd, np_[1:], ng_[1:], mb_[1:], lp_, lv_).find(lv_[1], "containment", 0.0) != []
