"""GPU parity of the Nodegraph bloom filter and the SBT search at the shapes where csrc/nodegraph.cu and the radix
sort under count_many change plan, and at the hash values and table sizes they special-case.

tests/test_gpu_nodegraph.py checks the same C ABI at small shapes, where every loop below runs once.  Here each
test crosses a threshold of the code -- a radix pass, a level of the scan under the sort, a grid-stride iteration,
a query block of sbt_find, the internal-node grid limit -- and asserts the shape fact, computed from the constants
mirrored below, that puts it past that threshold, so that a changed constant shows up as a failure rather than as a
test that quietly stops reaching its branch.  Every expected value comes from the CPU oracle (oracle/oracle.c),
whose batch calls and indexed SBT walk keep these sizes feasible.
"""
import ctypes as C

import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from util import splitmix64

pytestmark = pytest.mark.gpu

# csrc/sortops.cu
RS_TILE = 4096                # radix_sort_pairs: keys per sort block; the digit-count table has 256 entries per block
RADIX_BITS = 8                # one sort pass per 8 bits of the largest key
SCAN_TILE = 2048              # scan_exclusive_u64: elements per scan block; more recurse over the block totals
# csrc/nodegraph.cu
NG_THREADS = 256
SUM_BYTES_MAX_BLOCKS = 1024   # ng_sum_bytes_kernel grid
WORDS_MAX_BLOCKS = 2048       # ng_words_kernel grid (update, similarity, containment)
FIND_MAX_CELLS = 1 << 26      # sbt_find: a query block holds at most this many (node + leaf) x query cells ...
MAX_GRID_Y = 65535            # ... and at most this many queries; at most this many internal nodes per call
MAX_TABLES = 255
ERR_PANIC, ERR_INTERNAL = 1, 2

U64_MAX = (1 << 64) - 1
MAX_HASH = 1 << 63            # the sketches below are scaled (num = 0) with this max_hash


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


def sort_passes(total_bits):
    """count_many's radix passes: the largest key is the "bin already set" sentinel, total_bits itself."""
    return max(1, -(-total_bits.bit_length() // RADIX_BITS))


def sort_blocks(m):
    return -(-m // RS_TILE)


def scan_levels(m):
    """Recursion depth of the scan over the 256 x sort-blocks digit-count table of an m-key sort."""
    n, levels = 256 * sort_blocks(m), 0
    while n > SCAN_TILE:
        n, levels = -(-n // SCAN_TILE), levels + 1
    return levels


def words_grid(*graphs):
    """ng_words_kernel's grid for a pair of filters, from their summed table words."""
    w = max(sum((t + 31) // 32 for t in g) for g in graphs)
    return min(WORDS_MAX_BLOCKS, (w + NG_THREADS - 1) // NG_THREADS + 1)


def find_block_q(nq, n_nodes, n_leaves):
    return max(1, min(nq or 1, MAX_GRID_Y, FIND_MAX_CELLS // max(1, n_nodes + n_leaves)))


def u64(xs):
    return np.array([x % (1 << 64) for x in xs], dtype=np.uint64)


def same_state(g, o):
    assert g.tablesizes() == o.tablesizes()
    assert g.n_occupied_bins() == o.n_occupied_bins()
    assert g.unique_kmers() == o.unique_kmers()
    assert g.save() == o.save()


def count_both(g, o, batch):
    n_g, f_g = g.count_many(batch)
    n_o, f_o = o.count_many(batch)
    if not np.array_equal(f_g, f_o):
        bad = np.flatnonzero(f_g != f_o)
        raise AssertionError(f"is_new differs at {bad.size} positions, first {bad[:5].tolist()}: "
                             f"hashes {batch[bad[:5]].tolist()} got {f_g[bad[:5]].tolist()}")
    assert n_g == n_o == int(f_o.sum())


def get_both(g, o, probe):
    n_g, f_g = g.get_many(probe)
    n_o, f_o = o.get_many(probe)
    assert np.array_equal(f_g, f_o) and n_g == n_o


# ---- count_many at every radix-pass boundary ---------------------------------------------------------------
BOUNDARY_SETS = [
    [255], [100, 101, 54],
    [256], [100, 101, 55],
    [65535], [30011, 35524],
    [65536], [30011, 35525],
    [(1 << 24) - 1], [5000011, 6000000, 5777204],
    [1 << 24], [5000011, 6000000, 5777205],
    [1 << 32, 1000],
]
PASSES = {255: 1, 256: 2, 65535: 2, 65536: 3, (1 << 24) - 1: 3, 1 << 24: 4, (1 << 32) + 1000: 5}


def shared_bin_hashes(seed):
    """a and b of boundary_batch's pairs (a, a + len0) and (b + len0, b)"""
    r = splitmix64(seed, 12000)
    return int(r[0]) >> 1, int(r[1]) >> 1


def boundary_batch(ts, seed, already=()):
    """The hashes count_many special-cases, around random ones: hash 0 first, then the hashes `already` counted
    (their pairs sort as the "bin already set" sentinel), and len0 / k * len0 later (one clear bin, reached again
    past other tiles and past sentinels), the last bin of the last table, each table's len - 1 / len / k * len, a
    hash repeated more than RS_TILE pairs apart, and pairs of distinct hashes that share a bin in table 0 only, in
    both batch orders."""
    nt, l0 = len(ts), ts[0]
    r = splitmix64(seed, 12000)
    head = [0] + [int(x) for x in already] + [1, 1 << 63, U64_MAX, ts[-1] - 1]
    for t in ts:
        head += [t - 1, t, 3 * t, (U64_MAX // t) * t]
    a, b = shared_bin_hashes(seed)
    share = [a, a + l0, b + l0, b]  # same bin in table 0; apart in the other tables (l0 is no multiple of them)
    if nt > 1:
        assert all(a % t != (a + l0) % t for t in ts[1:]) and all(b % t != (b + l0) % t for t in ts[1:])
    rep = int(r[2])
    batch = u64(head + [rep] + share + r[3:6000].tolist() + [l0, rep, 5 * l0] + r[6000:].tolist() + [rep, 7 * l0])
    first, last = (batch == np.uint64(rep)).nonzero()[0][[0, -1]]
    assert (last - first) * nt > RS_TILE
    return batch


@pytest.mark.parametrize("ts", BOUNDARY_SETS, ids=lambda ts: "+".join(map(str, ts)))
def test_count_many_radix_pass_boundaries(ts):
    total = sum(ts)
    assert sort_passes(total) == PASSES[total]  # 5 is odd: the sorted keys come back from the temporaries
    if total & (total - 1) == 0:
        # the sentinel key alone needs the extra pass: a sort sized from bit_length(total - 1) is one short
        assert (total - 1).bit_length() % RADIX_BITS == 0
    g, o = smb.Nodegraph(ts, 21), orc.Nodegraph(ts, 21)
    # set some bins first, so that the main batch mixes clear keys with sentinels -- but few of them on small
    # tables, and none of the bins the main batch is built to decide: bin 0 and the shared bins of table 0, and
    # the last bin of the last table (key total_bits - 1, next to the sentinel)
    a, b = shared_bin_hashes(total)
    keep0 = {0, a % ts[0], b % ts[0]}
    seed_hashes = splitmix64(total + 1, min(300, total // 8))
    seed_hashes = np.array([h for h in seed_hashes if int(h) % ts[0] not in keep0 and int(h) % ts[-1] != ts[-1] - 1],
                           dtype=np.uint64)
    assert seed_hashes.size > 0
    count_both(g, o, seed_hashes)
    assert not any(o.bit(0, i) for i in keep0) and not o.bit(len(ts) - 1, ts[-1] - 1)
    batch = boundary_batch(ts, total, seed_hashes)
    count_both(g, o, batch)
    same_state(g, o)
    count_both(g, o, batch[::-1].copy())  # all seen: nothing new
    same_state(g, o)
    get_both(g, o, np.concatenate([batch[:3000], splitmix64(total + 2, 3000)]))


def test_count_many_scan_recursion_and_sum_grid():
    """10 M hashes x 7 tables in one call: a sort of more than 2^26 keys, whose digit-count scan recurses twice and
    whose is_new sum needs several grid-stride iterations; then a second batch on the same graph, where most bins
    are already set."""
    ts = [20000003, 20000023, 20000033, 20000047, 20000051, 20000069, 20000083]
    n = 10_000_000
    m = n * len(ts)
    assert 256 * sort_blocks(m) > SCAN_TILE * SCAN_TILE and scan_levels(m) == 2
    assert n > SUM_BYTES_MAX_BLOCKS * NG_THREADS
    g, o = smb.Nodegraph(ts, 21), orc.Nodegraph(ts, 21)
    h = splitmix64(77, n)
    h[n // 2:n // 2 + 1000] = h[:1000]  # repeats far apart
    count_both(g, o, h)
    same_state(g, o)
    h2 = np.concatenate([h[: n // 2], splitmix64(78, n // 2)])
    count_both(g, o, h2)
    same_state(g, o)
    get_both(g, o, np.concatenate([h[:100000], splitmix64(79, 100000)]))


# ---- ng_words_kernel past its first grid-stride iteration ------------------------------------------------------
LONG = (1 << 26) + 1   # 2^21 + 1 words: five grid-stride iterations of a 2048-block grid, the last of one word


def filled(ts, seed, n, keep=None):
    g, o = smb.Nodegraph(ts, 31), orc.Nodegraph(ts, 31)
    h = splitmix64(seed, n)
    if keep is not None:
        h = h[keep(h)]
    g.count_many(h)
    o.count_many(h)
    return g, o


def test_words_kernel_grid_stride():
    a_ts = [4099, LONG, 5003]                      # long table second, length = 1 mod 32
    b_ts = [4099, LONG + 30, 5003, 77]              # = 31 mod 32
    c_ts = [4099, 7001, (1 << 26) + (1 << 25)]      # long table third, = 0 mod 32
    for ts in (a_ts, b_ts, c_ts):  # the long table takes at least four grid-stride iterations
        assert max(ts) // 32 >= 4 * WORDS_MAX_BLOCKS * NG_THREADS
    assert {LONG % 32, (LONG + 30) % 32, c_ts[2] % 32} == {1, 31, 0}
    ga, oa = filled(a_ts, 1, 3_000_000)
    gb, ob = filled(b_ts, 2, 3_000_000)
    gc, oc = filled(c_ts, 3, 3_000_000)
    for (g1, o1), (g2, o2) in (((ga, oa), (gb, ob)), ((ga, oa), (gc, oc)), ((gb, ob), (gc, oc))):
        assert words_grid(g1.tablesizes(), g2.tablesizes()) == WORDS_MAX_BLOCKS
        for (x, ox), (y, oy) in (((g1, o1), (g2, o2)), ((g2, o2), (g1, o1))):
            assert x.similarity(y) == ox.similarity(oy)
            assert x.containment(y) == ox.containment(oy)

    # a shorter filter into a longer one
    gl, ol = filled([4099, LONG + 1000, 5003, 777], 4, 2_000_000)
    gs, os_ = filled([4099, LONG - 12345, 5003], 5, 2_000_000)
    gl.update(gs)
    ol.update(os_)
    same_state(gl, ol)
    # a longer `other` whose tail is clear
    gt, ot = filled([4099, LONG + 1000, 5003], 6, 2_000_000, keep=lambda h: h % np.uint64(LONG + 1000) < np.uint64(LONG))
    gself, oself = filled([4099, LONG, 5003], 7, 1_000_000)
    gself.update(gt)
    oself.update(ot)
    same_state(gself, oself)
    assert gself.similarity(gt) == oself.similarity(ot)

    # refused: the first set bit beyond self's table sits in a late grid-stride iteration of table 2 or 3;
    # the tables before it and its in-range bits are put, as the reference's loop puts them before it panics
    self_ts = [4099, LONG, LONG]
    for other_ts in ([4099, LONG + 3000, LONG + 3000], [4099, LONG, LONG + 3000]):
        gx, ox = filled(self_ts, 8, 500_000)
        go, oo = filled(other_ts, 9, 2_000_000)
        assert words_grid(self_ts, other_ts) == WORDS_MAX_BLOCKS
        assert (LONG // 32) // (WORDS_MAX_BLOCKS * NG_THREADS) == 4  # the words beyond self's table: fifth iteration
        with pytest.raises(smb.SourmashError) as e:
            gx.update(go)
        assert e.value.code == ERR_PANIC
        with pytest.raises(orc.SourmashError):
            ox.update(oo)
        same_state(gx, ox)


# ---- small tables, table counts, refusals ------------------------------------------------------------------------
def test_table_count_and_size_refusals():
    ts = np.full(MAX_TABLES + 1, 7, dtype=np.uint64)
    L = smb.lib()
    for n, sizes, code, msg in ((MAX_TABLES + 1, ts, ERR_INTERNAL, None),
                                (3, u64([5, 0, 7]), ERR_PANIC,
                                 "sourmash panicked: attempt to calculate the remainder with a divisor of zero")):
        L.sourmash_err_clear()
        p = L.smgpu_nodegraph_new(smb._vp(sizes), n, 21)
        assert not p
        with pytest.raises(smb.SourmashError) as e:
            smb.Nodegraph(sizes[:n], 21)
        assert e.value.code == code
        if msg:
            assert e.value.message == msg
    g = smb.Nodegraph(ts[:MAX_TABLES], 21)  # the largest accepted count
    assert len(g.tablesizes()) == MAX_TABLES


def test_device_resident_count_and_get():
    torch = pytest.importorskip("torch")
    ts = [1009, 70001, 125598]
    g, o = smb.Nodegraph(ts, 21), orc.Nodegraph(ts, 21)
    batch = boundary_batch(ts, 5)
    d_h = torch.from_numpy(batch.view(np.int64)).cuda()
    d_new = torch.full((batch.size,), 0xAB, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()  # the library works on its own stream, which does not wait for torch's
    n = smb._call("smgpu_nodegraph_count_many", g._p, d_h.data_ptr(), batch.size, d_new.data_ptr(), True)
    n_o, f_o = o.count_many(batch)
    assert n == n_o and np.array_equal(d_new.cpu().numpy(), f_o.astype(np.uint8))
    same_state(g, o)
    probe = np.concatenate([batch[:2000], splitmix64(6, 2000)])
    d_p = torch.from_numpy(probe.view(np.int64)).cuda()
    d_present = torch.full((probe.size,), 0xAB, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    n = smb._call("smgpu_nodegraph_get_many", g._p, d_p.data_ptr(), probe.size, d_present.data_ptr(), True)
    n_o, f_o = o.get_many(probe)
    assert n == n_o and np.array_equal(d_present.cpu().numpy(), f_o)


def test_no_tables_writes_every_output():
    """A graph with no tables: count() is 0 and get() is 1 for every hash; both outputs are written in full."""
    torch = pytest.importorskip("torch")
    g, o = smb.Nodegraph([], 21), orc.Nodegraph([], 21)
    h = u64([0, 1, 5, U64_MAX] + splitmix64(3, 1000).tolist())
    n_new, want_new = o.count_many(h)
    n_hit, want_present = o.get_many(h)
    assert n_new == 0 and not want_new.any() and n_hit == h.size and want_present.all()
    L = smb.lib()
    for fn, want, n_want in (("smgpu_nodegraph_count_many", want_new, n_new),
                             ("smgpu_nodegraph_get_many", want_present, n_hit)):
        out = np.full(h.size, 0xAB, dtype=np.uint8)
        L.sourmash_err_clear()
        n = getattr(L, fn)(g._p, smb._vp(h), h.size, smb._vp(out), False)
        assert L.sourmash_err_get_last_code() == 0
        assert n == n_want and np.array_equal(out, want.astype(np.uint8)), fn
        d_h = torch.from_numpy(h.view(np.int64)).cuda()
        d_out = torch.full((h.size,), 0xAB, dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()  # the library works on its own stream, which does not wait for torch's
        n = smb._call(fn, g._p, d_h.data_ptr(), h.size, d_out.data_ptr(), True)
        assert n == n_want and np.array_equal(d_out.cpu().numpy(), want.astype(np.uint8)), fn
    same_state(g, o)


# ---- SBT search ---------------------------------------------------------------------------------------------------
def sketch_pair(hashes):
    hs = np.unique(np.asarray(hashes, dtype=np.uint64) % np.uint64(MAX_HASH))
    o = orc.KmerMinHash(0, 31, False, 42, MAX_HASH)
    o.add_many(hs)
    return o.mins_np(), o


def csr(rows):
    offs = np.zeros(len(rows) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([r.size for r in rows])
    flat = np.concatenate(rows) if rows else np.zeros(0, dtype=np.uint64)
    return smb.SketchCollection.from_csr(flat, offs, len(rows), 0, 31, 42, MAX_HASH)


def raw_find(d, npos, gnodes, mnb, lpos, leaves, queries, mode, thr, with_offsets=True, cap=None):
    """smgpu_sbt_find with node arrays given as lists (positions may repeat), outputs preset to garbage.
    Returns (code, total, offsets or None, hits buffer)."""
    nq = len(queries)
    a_np = np.ascontiguousarray(npos, dtype=np.uint64)
    a_ng = (C.c_void_p * max(1, len(gnodes)))(*[g._p for g in gnodes])
    a_mb = np.ascontiguousarray(mnb, dtype=np.uint64)
    a_lp = np.ascontiguousarray(lpos, dtype=np.uint64)
    offs = np.full(nq + 1, 0xDEAD, dtype=np.uint64)
    hits = np.full(max(1, cap or 0), 0xBEEF, dtype=np.uint64)
    L = smb.lib()
    L.sourmash_err_clear()
    total = L.smgpu_sbt_find(d, smb._vp(a_np), C.cast(a_ng, C.c_void_p), smb._vp(a_mb), len(npos), smb._vp(a_lp), leaves._p,
                             queries._p, 1 if mode == "containment" else 0, thr, smb._vp(offs) if with_offsets else None,
                             smb._vp(hits) if cap is not None else None, cap or 0)
    code = L.sourmash_err_get_last_code()
    L.sourmash_err_clear()
    return code, total, (offs if with_offsets else None), hits


def under(a, pos, d):
    while pos:
        pos = (pos - 1) // d
        if pos == a:
            return True
    return False


class SmallTree:
    """A random heap-layout tree (as in test_gpu_nodegraph.test_sbt_find_random_trees): leaves in clusters that
    share hashes, internal nodes holding everything below them, a hole, a node with a tiny min_n_below."""

    def __init__(self, d=3, n_leaves=20, seed=11):
        self.d = d
        pool = splitmix64(seed, 8000)
        n_internal = 1
        while n_internal * (d - 1) + 1 < n_leaves:
            n_internal += 1
        self.lpos = list(range(n_internal, n_internal + n_leaves))
        del self.lpos[3]
        self.leaf_rows, self.o_leaves = [], []
        for j in range(len(self.lpos)):
            cl = j // 3
            row, o = sketch_pair(np.concatenate([pool[j * 97 % 3000:j * 97 % 3000 + 120], pool[3000 + cl * 150:3150 + cl * 150]]))
            self.leaf_rows.append(row)
            self.o_leaves.append(o)
        self.leaves = csr(self.leaf_rows)
        ts = [4999, 5003, 5009]
        self.npos, self.gnodes, self.onodes, self.mnb = [], [], [], []
        for p in range(n_internal):
            if p == 2:
                continue
            below = [i for i, l in enumerate(self.lpos) if under(p, l, d)]
            g, o = smb.Nodegraph(ts, 31), orc.Nodegraph(ts, 31)
            for i in below:
                g.count_many(self.leaf_rows[i])
                o.count_many(self.leaf_rows[i])
            self.npos.append(p)
            self.gnodes.append(g)
            self.onodes.append(o)
            self.mnb.append(1 if p == 1 else max(1, min([self.leaf_rows[i].size for i in below] or [1])))
        self.pool = pool

    def oracle(self, npos=None, onodes=None, mnb=None, lpos=None, o_leaves=None):
        return orc.SbtOracle(self.d, self.npos if npos is None else npos, self.onodes if onodes is None else onodes,
                             self.mnb if mnb is None else mnb, self.lpos if lpos is None else lpos,
                             self.o_leaves if o_leaves is None else o_leaves)

    def query_sketches(self, n):
        """n distinct sketches: parts of leaves plus noise; the last is empty."""
        out = []
        for j in range(n - 1):
            src = self.leaf_rows[(j * 5) % len(self.leaf_rows)]
            extra = self.pool[4000 + (j * 311) % 3500:4000 + (j * 311) % 3500 + 10 + j]
            out.append(sketch_pair(np.concatenate([src[: max(1, src.size * (j % 7 + 1) // 8)], extra])))
        out.append(sketch_pair([]))
        return out


@pytest.fixture(scope="module")
def small_tree():
    return SmallTree()


def test_sbt_find_two_query_blocks(small_tree):
    t = small_tree
    sk = t.query_sketches(40)
    nq = 70_001
    block_q = find_block_q(nq, len(t.npos), len(t.lpos))
    assert block_q == MAX_GRID_Y and -(-nq // block_q) == 2
    idx = (splitmix64(21, nq) % np.uint64(len(sk) - 1)).astype(np.int64)
    for row, s in ((0, 3), (MAX_GRID_Y - 1, 0), (MAX_GRID_Y, len(sk) - 1), (MAX_GRID_Y + 1, 5), (nq - 1, 7)):
        idx[row] = s
    assert sk[len(sk) - 1][0].size == 0 and idx[MAX_GRID_Y] == len(sk) - 1
    queries = csr([sk[i][0] for i in idx])
    tree = t.oracle()
    n_hits = 0
    for mode in ("similarity", "containment"):
        for thr in (0.0, 0.2):
            want = [tree.find(o, mode, thr) for _, o in sk]
            got = smb.sbt_find(t.d, dict(zip(t.npos, zip(t.gnodes, t.mnb))), t.lpos, t.leaves, queries, mode, thr)
            assert len(got) == nq
            bad = [q for q in range(nq) if got[q] != want[idx[q]]]
            assert not bad, (mode, thr, len(bad), bad[:5])
            n_hits += sum(len(w) for w in want)
            assert not got[MAX_GRID_Y]  # the empty sketch
            assert any(got[:MAX_GRID_Y]) and any(got[MAX_GRID_Y:])
    assert n_hits > 0


def test_sbt_find_65535_nodes():
    """The largest node grid sbt_matches_kernel takes, with more query blocks than one: d = 256, a root, 256
    level-1 nodes and level-2 nodes up to 65 535 nodes, one leaf under each level-2 node.  The filters are sized so
    that a query passes only the paths its hashes come from."""
    d = 256
    n_nodes = MAX_GRID_Y
    lvl2 = list(range(d + 1, d + 1 + n_nodes - 1 - d))
    npos = [0] + list(range(1, d + 1)) + lvl2
    assert len(npos) == n_nodes and npos == sorted(npos)
    lpos = [d * p + 1 for p in lvl2]
    n_leaves = len(lpos)
    per = 6
    pool = splitmix64(31, n_leaves * per) % np.uint64(MAX_HASH)
    rows = [np.sort(pool[i * per:(i + 1) * per]) for i in range(n_leaves)]
    o_leaves = []
    for r in rows:
        o = orc.KmerMinHash(0, 31, False, 42, MAX_HASH)
        o.add_many(r)
        o_leaves.append(o)
    leaves = csr(rows)
    # node contents: level 2 = its leaf, level 1 = its level-2 children's leaves, root = everything
    leaf_of = {p: i for i, p in enumerate(lvl2)}
    onodes, gnodes, mnb = [], [], []
    for p in npos:
        if p == 0:
            hs, ts = pool, [4000037, 4000039]
        elif p <= d:
            kids = [leaf_of[c] for c in range(d * p + 1, d * p + d + 1) if c in leaf_of]
            hs = np.concatenate([rows[i] for i in kids]) if kids else np.zeros(0, dtype=np.uint64)
            ts = [40009, 40013]
        else:
            hs, ts = rows[leaf_of[p]], [211, 223]
        o = orc.Nodegraph(ts, 31)
        o.count_many(hs)
        onodes.append(o)
        gnodes.append(smb.Nodegraph.from_buffer(o.save()))
        mnb.append(per)
    # queries: the hashes of one leaf whose level-2 node is among the last 1 000 entries, of one other leaf, and noise
    nq = 1200
    block_q = find_block_q(nq, n_nodes, n_leaves)
    n_blocks = -(-nq // block_q)
    assert block_q < nq and n_blocks >= 3 and nq % block_q != 0
    r = splitmix64(32, 3 * nq)
    tail_leaf = [leaf_of[npos[n_nodes - 1 - int(x) % 1000]] for x in r[:nq]]
    other_leaf = [int(x) % n_leaves for x in r[nq:2 * nq]]
    sk = [sketch_pair(np.concatenate([rows[tail_leaf[q]], rows[other_leaf[q]][:4], r[2 * nq + q:2 * nq + q + 1]]))
          for q in range(nq)]
    queries = csr([s[0] for s in sk])
    tree = orc.SbtOracle(d, npos, onodes, mnb, lpos, o_leaves)
    gdict = dict(zip(npos, zip(gnodes, mnb)))
    tail_leaves = {lpos[leaf_of[p]] for p in npos[n_nodes - 1000:]}
    for mode, thr in (("similarity", 0.1), ("containment", 0.3)):
        got = smb.sbt_find(d, gdict, lpos, leaves, queries, mode, thr)
        for q in range(nq):
            assert got[q] == tree.find(sk[q][1], mode, thr), (mode, thr, q)
        # the walk reaches the last 1 000 node entries for queries of every block
        for b in range(n_blocks):
            assert any(tail_leaves.intersection(got[q]) for q in range(b * block_q, min(nq, (b + 1) * block_q))), b
    # one node more is refused, but only once there is a query to run it for
    extra_pos = npos + [d * lvl2[-1] + 2]
    extra_nodes = gnodes + [smb.Nodegraph([211, 223], 31)]
    code, total, _, _ = raw_find(d, extra_pos, extra_nodes, mnb + [per], lpos, leaves, queries, "similarity", 0.1)
    assert code == ERR_INTERNAL
    code, total, offs, _ = raw_find(d, extra_pos, extra_nodes, mnb + [per], lpos, leaves, csr([]), "similarity", 0.1)
    assert code == 0 and total == 0 and offs.tolist() == [0]


def test_sbt_find_edges(small_tree):
    t = small_tree
    sk = t.query_sketches(12)
    queries = csr([s[0] for s in sk])
    tree = t.oracle()
    want = [tree.find(o, "containment", 0.05) for _, o in sk]
    flat = [h for w in want for h in w]
    want_offs = np.cumsum([0] + [len(w) for w in want])
    assert len(flat) > 10
    args = (t.d, t.npos, t.gnodes, t.mnb, t.lpos, t.leaves, queries, "containment", 0.05)
    # hits_cap below the total: the first hits_cap hits in walk order, the whole total and complete offsets
    for cap in (0, 1, len(flat) // 2, len(flat) - 1, len(flat), len(flat) + 5):
        code, total, offs, hits = raw_find(*args, cap=cap)
        assert code == 0 and total == len(flat)
        assert offs.tolist() == want_offs.tolist()
        k = min(cap, total)
        assert hits[:k].tolist() == flat[:k] and (hits[k:] == 0xBEEF).all()
    # no offsets
    code, total, offs, hits = raw_find(*args, with_offsets=False, cap=len(flat))
    assert code == 0 and total == len(flat) and hits.tolist() == flat
    # no queries
    code, total, offs, hits = raw_find(*args[:6], csr([]), "containment", 0.05, cap=4)
    assert code == 0 and total == 0 and offs.tolist() == [0] and (hits == 0xBEEF).all()
    # no internal nodes, a leaf at the root
    for j in (0, 4):
        leaf = csr([t.leaf_rows[j]])
        code, total, offs, hits = raw_find(t.d, [], [], [], [0], leaf, queries, "similarity", 0.0, cap=len(sk))
        o1 = orc.SbtOracle(t.d, [], [], [], [0], [t.o_leaves[j]])
        w = [o1.find(o, "similarity", 0.0) for _, o in sk]
        assert code == 0 and offs.tolist() == np.cumsum([0] + [len(x) for x in w]).tolist()
        assert hits[:total].tolist() == [h for x in w for h in x] and total > 0
    # min_n_below = 0: matches / 0 is inf (taken) or NaN (not taken), as the oracle computes it
    mnb0 = [0 if p in (0, 4) else m for p, m in zip(t.npos, t.mnb)]
    o0 = t.oracle(mnb=mnb0)
    for thr in (0.0, 0.5):
        w = [o0.find(o, "similarity", thr) for _, o in sk]
        code, total, offs, hits = raw_find(t.d, t.npos, t.gnodes, mnb0, t.lpos, t.leaves, queries, "similarity", thr,
                                           cap=sum(map(len, w)))
        assert code == 0 and offs.tolist() == np.cumsum([0] + [len(x) for x in w]).tolist()
        assert hits[:total].tolist() == [h for x in w for h in x]
    # a node position listed twice (the first entry wins), each way round
    empty_g, empty_o = smb.Nodegraph([4999, 5003, 5009], 31), orc.Nodegraph([4999, 5003, 5009], 31)
    i1 = t.npos.index(1)
    for npos, gn, on, mb in ((t.npos + [1], t.gnodes + [empty_g], t.onodes + [empty_o], t.mnb + [1]),
                             ([1] + t.npos, [empty_g] + t.gnodes, [empty_o] + t.onodes, [1] + t.mnb),
                             (t.npos[:i1 + 1] + [1] + t.npos[i1 + 1:], t.gnodes[:i1 + 1] + [empty_g] + t.gnodes[i1 + 1:],
                              t.onodes[:i1 + 1] + [empty_o] + t.onodes[i1 + 1:], t.mnb[:i1 + 1] + [1] + t.mnb[i1 + 1:])):
        od = t.oracle(npos=npos, onodes=on, mnb=mb)
        for mode in ("similarity", "containment"):
            w = [od.find(o, mode, 0.05) for _, o in sk]
            code, total, offs, hits = raw_find(t.d, npos, gn, mb, t.lpos, t.leaves, queries, mode, 0.05, cap=sum(map(len, w)))
            assert code == 0 and offs.tolist() == np.cumsum([0] + [len(x) for x in w]).tolist()
            assert hits[:total].tolist() == [h for x in w for h in x]
