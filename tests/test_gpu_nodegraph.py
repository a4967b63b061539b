"""GPU parity tests for the Nodegraph bloom filter and the SBT search (SURVEY 8(f) rank 3): the C ABI
(smgpu_nodegraph_*, smgpu_sbt_find) against the CPU oracle and the reference's own fixtures
(src/index/nodegraph.rs:236-821, src/index/sbt.rs:526-590)."""
import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from util import golden, sbt_v5_tree, splitmix64

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


def _sketch_pair(sk):
    args = (0 if sk["max_hash"] else sk["num"], sk["ksize"], sk["molecule"] == "protein", sk["seed"], sk["max_hash"], False)
    g, o = smb.KmerMinHash(*args), orc.KmerMinHash(*args)
    g.set_mins(np.asarray(sk["mins"], dtype=np.uint64))
    o.add_many(sk["mins"])
    return g, o


def _same_state(g, o):
    assert g.tablesizes() == o.tablesizes()
    assert g.ksize() == o.ksize()
    assert g.n_occupied_bins() == o.n_occupied_bins()
    assert g.unique_kmers() == o.unique_kmers()
    assert g.save() == o.save()


# ---- the reference's own tests ----------------------------------------------------------------------
def test_count_and_get():  # nodegraph.rs:236-254
    g = smb.Nodegraph([10], 3)
    assert g.count(801084876663808) is True
    assert g.get(801084876663808) == 1 and g.unique_kmers() == 1
    assert g.count(801084876663808) is False and g.unique_kmers() == 1
    for h in (0, 1, 9, 10, 2**64 - 1, 0x123456789ABCDEF):
        g = smb.Nodegraph([10], 3)
        g.count(h)
        assert g.get(h) == 1


def test_load_save_roundtrip_and_fixture_hashes():  # nodegraph.rs:256-279, 292-821
    d, nodes, leaf_positions, t = sbt_v5_tree()
    for p, (raw, _) in nodes.items():
        g = smb.Nodegraph.from_buffer(raw)
        assert g.save() == raw
        _same_state(g, orc.Nodegraph.from_buffer(raw))
    spec = t["load_nodegraph"]
    g = smb.Nodegraph.from_buffer(nodes[0][0])
    assert g.tablesizes() == spec["tablesizes"]
    n, flags = g.get_many(spec["absent"])
    assert n == 0 and not flags.any()
    n, flags = g.get_many(spec["present"])
    assert n == 500 and flags.all()


def test_update_fixture():  # nodegraph.rs:271-290
    d, nodes, leaf_positions, t = sbt_v5_tree()
    g0 = smb.Nodegraph([99991, 99989, 99971, 99961], 1)
    g0.update(smb.Nodegraph.from_buffer(nodes[1][0]))
    g0.update(smb.Nodegraph.from_buffer(nodes[2][0]))
    parent = smb.Nodegraph.from_buffer(nodes[0][0])
    assert g0.save()[19:] == nodes[0][0][19:]
    assert g0.similarity(parent) == 1.0
    o0, o1 = orc.Nodegraph.from_buffer(nodes[0][0]), orc.Nodegraph.from_buffer(nodes[1][0])
    g1 = smb.Nodegraph.from_buffer(nodes[1][0])
    assert parent.similarity(g1) == o0.similarity(o1) and parent.containment(g1) == o0.containment(o1)
    assert g1.similarity(parent) == o1.similarity(o0) and g1.containment(parent) == o1.containment(o0)


def test_bad_file_images():
    d, nodes, leaf_positions, t = sbt_v5_tree()
    raw = nodes[0][0]
    for bad in (raw[:10], b"OXLJ" + raw[4:], raw[:4] + b"\x03" + raw[5:], raw[:5] + b"\x01" + raw[6:], raw[:-5]):
        with pytest.raises(smb.SourmashError) as e:
            smb.Nodegraph.from_buffer(bad)
        assert e.value.code == 1
        with pytest.raises(orc.SourmashError):
            orc.Nodegraph.from_buffer(bad)


def test_sbt_find_fixture():  # sbt.rs:543-551 (tree) next to :566-588 (the same queries through LinearIndex)
    d, nodes, leaf_positions, t = sbt_v5_tree()
    leaves_json = golden("sbt_v5_leaves.json")["leaves"]
    g_nodes = {p: (smb.Nodegraph.from_buffer(raw), mnb) for p, (raw, mnb) in nodes.items()}
    o_nodes = {p: (orc.Nodegraph.from_buffer(raw), mnb) for p, (raw, mnb) in nodes.items()}
    coll = smb.SketchCollection()
    o_leaves = {}
    for p in leaf_positions:
        g, o = _sketch_pair(leaves_json[str(p)]["sketch"])
        coll.push(g)
        o_leaves[p] = o
    want = t["asserted_sbt_find"]
    q = leaf_positions.index(want["query_position"])
    for mode in ("similarity", "containment"):
        for thr in (0.5, 0.1, 0.0, 0.9):
            got = smb.sbt_find(d, g_nodes, leaf_positions, coll, coll, mode, thr)
            for qi, p in enumerate(leaf_positions):
                assert got[qi] == orc.sbt_find(d, o_nodes, o_leaves, o_leaves[p], mode, thr), (mode, thr, p)
            if mode == "similarity" and thr in (0.5, 0.1):
                assert len(got[q]) == want["similarity@%s" % thr]
    # Node<Nodegraph> x Leaf<Signature> numerators
    for p, (ng, mnb) in g_nodes.items():
        for lp in leaf_positions:
            g, o = _sketch_pair(leaves_json[str(lp)]["sketch"])
            assert ng.matches(g) == o_nodes[p][0].matches(o)


# ---- randomised parity ------------------------------------------------------------------------------
@pytest.mark.parametrize("tablesizes", [[10], [31, 32, 33], [64, 96, 8], [997, 1009, 1013, 1019], [1, 2, 3], [40000, 39989], [255] * 7,
                                        [1], [2], [32], [63, 64, 65], [1023, 1024, 1025, 4095, 4096, 4097],
                                        list(range(1, 256))])
def test_count_get_random(tablesizes):
    r = splitmix64(sum(tablesizes) + len(tablesizes), 4000)
    g, o = smb.Nodegraph(tablesizes, 21), orc.Nodegraph(tablesizes, 21)
    for lo, hi in ((0, 1), (1, 50), (50, 1500), (1500, 4000)):
        batch = np.concatenate([r[lo:hi], r[lo:hi][::3], r[:lo][:40]])  # repeats inside the batch and of earlier batches
        n_new, flags = g.count_many(batch)
        want = [o.count(int(h)) for h in batch]
        assert list(flags) == want and n_new == sum(want)
        _same_state(g, o)
    probe = np.concatenate([r[:500], splitmix64(99, 500)])
    n, flags = g.get_many(probe)
    want = [o.get(int(h)) for h in probe]
    assert list(flags) == want and n == sum(want)
    # save -> load reproduces the filter (tables whose length is a multiple of 8 are one byte short on
    # save against what from_reader expects, nodegraph.rs:110-127 vs :154: both sides must fail alike)
    img = o.save()
    try:
        o2 = orc.Nodegraph.from_buffer(img)
    except orc.SourmashError:
        with pytest.raises(smb.SourmashError):
            smb.Nodegraph.from_buffer(img)
    else:
        g2 = smb.Nodegraph.from_buffer(img)
        assert g2.save() == o2.save() and g2.n_occupied_bins() == o2.n_occupied_bins() and g2.unique_kmers() == 0


def test_update_similarity_containment_random():
    ts = [997, 1009, 1013]
    r = splitmix64(5, 3000)
    ga, oa = smb.Nodegraph(ts, 31), orc.Nodegraph(ts, 31)
    gb, ob = smb.Nodegraph(ts, 31), orc.Nodegraph(ts, 31)
    ga.count_many(r[:300]); [oa.count(int(h)) for h in r[:300]]
    gb.count_many(r[200:700]); [ob.count(int(h)) for h in r[200:700]]
    assert ga.similarity(gb) == oa.similarity(ob) and gb.similarity(ga) == ob.similarity(oa)
    assert ga.containment(gb) == oa.containment(ob) and gb.containment(ga) == ob.containment(oa)
    ga.update(gb); oa.update(ob)
    _same_state(ga, oa)
    assert ga.similarity(gb) == oa.similarity(ob)
    # empty against empty: 0 / 0
    ge, oe = smb.Nodegraph(ts, 31), orc.Nodegraph(ts, 31)
    assert np.isnan(ge.similarity(ge)) and np.isnan(oe.similarity(oe))
    assert ge.containment(ge) == 0.0 == oe.containment(oe)
    # a shorter filter folds into a longer one; the other way round is refused
    gs, os_ = smb.Nodegraph([500, 600], 31), orc.Nodegraph([500, 600], 31)
    gs.count_many(r[:100]); [os_.count(int(h)) for h in r[:100]]
    ga.update(gs); oa.update(os_)
    _same_state(ga, oa)
    with pytest.raises(smb.SourmashError):
        gs.update(ga)
    with pytest.raises(orc.SourmashError):
        os_.update(oa)
    _same_state(gs, os_)          # what was put before the first out-of-range bit stays (the panic comes mid-loop)
    # a LONGER table on the other side is fine while no set bit lies beyond self's table (FixedBitSet::put
    # only panics on the bit it is handed)
    gl, ol = smb.Nodegraph([2000, 2003], 31), orc.Nodegraph([2000, 2003], 31)
    low = [int(h) for h in r[:400] if int(h) % 2000 < 500 and int(h) % 2003 < 600]
    assert len(low) > 5
    gl.count_many(low); [ol.count(h) for h in low]
    g5, o5 = smb.Nodegraph([500, 600], 31), orc.Nodegraph([500, 600], 31)
    g5.update(gl); o5.update(ol)
    _same_state(g5, o5)
    assert g5.n_occupied_bins() == 0 and sum(g5.get_many(low)[1]) > 0


@pytest.mark.parametrize("d,n_leaves,num,mx", [(2, 13, 200, 0), (3, 20, 0, 2**64 // 2000), (2, 1, 50, 0), (4, 9, 64, 0)])
def test_sbt_find_random_trees(d, n_leaves, num, mx):
    """Random trees in heap layout: leaves in clusters that share hashes, internal nodes = bloom filters over
    everything below them (as `sourmash index` builds them), plus holes, a node with a tiny min_n_below and an
    empty query."""
    rng = splitmix64(1000 * d + n_leaves, 64)
    n_internal = 1
    while n_internal * (d - 1) + 1 < n_leaves:  # enough internal nodes so that every leaf has a parent
        n_internal += 1
    first_leaf = n_internal
    leaf_positions = list(range(first_leaf, first_leaf + n_leaves))
    if n_leaves > 4:
        del leaf_positions[3]  # a hole: that position is neither node nor leaf
    pool = splitmix64(7 + n_leaves, 6000)
    if mx:
        pool = pool % np.uint64(mx)
    g_leaves, o_leaves, coll = {}, {}, smb.SketchCollection()
    for j, p in enumerate(leaf_positions):
        cl = j // 3
        own = pool[(j * 97) % 3000:(j * 97) % 3000 + 120]
        shared = pool[3000 + cl * 150:3000 + cl * 150 + 150]
        hs = np.unique(np.concatenate([own, shared]))
        g, o = smb.KmerMinHash(num, 31, False, 42, mx, False), orc.KmerMinHash(num, 31, False, 42, mx, False)
        for h in hs:
            o.add_hash(int(h))
        g.set_mins(o.mins_np())
        g_leaves[p], o_leaves[p] = g, o
        coll.push(g)
    ts = [4999, 5003, 5009]
    g_nodes, o_nodes = {}, {}
    for p in range(n_internal):
        if p == 2 and n_internal > 4:
            continue  # a missing internal node prunes its subtree
        below = [l for l in leaf_positions if _under(p, l, d)]
        g, o = smb.Nodegraph(ts, 31), orc.Nodegraph(ts, 31)
        for l in below:
            g.count_many(o_leaves[l].mins_np())
            for h in o_leaves[l].mins:
                o.count(h)
        mnb = 1 if p == 1 else max(1, min([o_leaves[l].size() for l in below] or [1]))
        g_nodes[p], o_nodes[p] = (g, mnb), (o, mnb)
    queries = smb.SketchCollection()
    o_queries = []
    for j in range(6):
        g, o = smb.KmerMinHash(num, 31, False, 42, mx, False), orc.KmerMinHash(num, 31, False, 42, mx, False)
        if j < 5:
            src = o_leaves[leaf_positions[(j * 5) % len(leaf_positions)]].mins_np()
            extra = pool[(j * 311) % 2500:(j * 311) % 2500 + 60]
            for h in np.concatenate([src[: len(src) * (j + 1) // 6], extra]):
                o.add_hash(int(h))
            g.set_mins(o.mins_np())
        queries.push(g)
        o_queries.append(o)
    for mode in ("similarity", "containment"):
        for thr in (0.0, 0.05, 0.3, 0.8):
            got = smb.sbt_find(d, g_nodes, leaf_positions, coll, queries, mode, thr)
            for qi, oq in enumerate(o_queries):
                assert got[qi] == orc.sbt_find(d, o_nodes, o_leaves, oq, mode, thr), (mode, thr, qi)


def _under(a, pos, d):
    while pos:
        pos = (pos - 1) // d
        if pos == a:
            return True
    return False
