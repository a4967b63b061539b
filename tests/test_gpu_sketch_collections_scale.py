"""smgpu_sketch_collections (csrc/sketch_many.cu) past the thresholds where its plan changes, bit for bit against the
oracle loop
    for s in sequences: for t in templates: mh = KmerMinHash(t); mh.add_sequence(s, True); rows[t].append(mh.mins)

tests/test_gpu_sketch_collections.py checks the same call at shapes where every grid-stride loop runs once, the
survivor scan recurses at most once, sequence ids sort in one radix pass and only template 0 of a fused trio ever
overflows its survivor region.  Here each test crosses one of those thresholds -- the exact end of a survivor
region, each re-run shape, a radix pass over sequence ids, a level of the survivor scan, the persistent sketch grid
and its shared tile counter, rows cut short under an estimated threshold, empty results, calls of changing shape on
one context -- and asserts the shape fact, computed from the constants mirrored below and from the oracle, that puts
it there, so that a changed constant fails the test instead of quietly skipping the branch.  Where the branch is the
point of the test, the launch counts confirm it ran: the sketch launches per kernel from the profiler (one stream),
and every launch of the call from smb.launch_count() where the protein kernels are involved, against a model of the
call's launches.  Profiled calls run once more unprofiled, and both must equal the oracle."""
import contextlib
import os

import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from test_gpu_sketch_collections import dirty, offsets_of, polya_input
from util import MAX_HASH_1000, random_dna, splitmix64

pytestmark = pytest.mark.gpu

# csrc/sortops.cu
SCAN_TILE = 2048                 # scan_exclusive_u64: elements per scan block; more recurse over the block totals
RS_TILE = 4096                   # radix_sort_pairs: keys per sort block; its digit-count table has 256 per block
RADIX_BITS = 8                   # one sort pass per 8 bits of the largest key
# csrc/sketch_many.cu
MANY_THREADS = 148 * 16 * 256    # grid_for: the grid of pos_to_seq / flags / seg_base / keep / compact is capped here
MAX_TEMPLATES = 6
# csrc/protein.cu
PROTEIN_THREADS = 148 * 32 * 256  # protein_blocks: the grid of translate / compact / hash is capped here
# csrc/kernels.cuh
SK_TILE = 4096                   # window starts per tile of the sketch kernels
SK_CTAS_PER_SM = 5               # persistent CTAs per SM of the fast-path (k = 21, 31, 51) kernels

U64_MAX = 2**64 - 1
KINDS = ("sketch_k21", "sketch_k31", "sketch_k51", "sketch_other", "sketch_multi")
NT = os.cpu_count() or 4


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


# ------------------------------------------------------------------------------------------------
# mirrors of the host logic of sketch_collections
# ------------------------------------------------------------------------------------------------
def bits_of(x):
    """sketch_many.cu bits_of: the radix sort's end bit for keys up to x"""
    return max(1, int(x).bit_length())


def sort_passes(bits):
    return min(8, max(1, -(-bits // RADIX_BITS)))


def threshold(p, lens):
    """(thr, frac) of template p = (num, k, prot, seed, max_hash) over sequences of lengths `lens`"""
    num, k, prot, seed, mx = p
    if mx:
        return mx, float(mx) / 18446744073709551616.0
    median = float(max(1, sorted(lens)[len(lens) // 2]))
    frac = min(1.0, 16.0 * float(num) / (2.0 * median if prot else median))
    return (int(frac * 18446744073709551616.0) if frac < 1.0 else U64_MAX), frac


def windows_of(p, lens):
    """the survivor reservation's window count: n for DNA, protein_slots = 2n + 6 n_seqs for protein"""
    return 2 * sum(lens) + 6 * len(lens) if p[2] else sum(lens)


def cap_of(p, lens):
    """cap = (uint64_t)(frac * 1.25 * (double)windows) + 4096, evaluated in double in the C++ order"""
    _, frac = threshold(p, lens)
    return int(frac * 1.25 * float(windows_of(p, lens))) + 4096


def scan_launches(n):
    if n == 0:
        return 0
    if n <= SCAN_TILE:
        return 1
    return 2 + scan_launches(-(-n // SCAN_TILE))


def scan_levels(n):
    levels = 0
    while n > SCAN_TILE:
        n, levels = -(-n // SCAN_TILE), levels + 1
    return levels


def sort_launches(n, bits):
    if n < 2:
        return 0
    return sort_passes(bits) * (2 + scan_launches(256 * -(-n // RS_TILE)))


def group_launches(count, n_seqs, thr):
    """group_survivors: pos_to_seq, the sorts by hash and by sequence, flags, scan, seg_base, keep, scan, compact"""
    if count == 0:
        return 0
    return 5 + sort_launches(count, bits_of(thr)) + sort_launches(count, bits_of(n_seqs)) + 2 * scan_launches(count)


def translate_launches(lens):
    """the shared six-frame translation: translate, scan over the slots, compact, sequence starts"""
    slots = 2 * sum(lens) + 6 * len(lens)
    return 3 + scan_launches(slots + 1) if sum(lens) else 0


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def counted():
    """Per-kernel sketch launch counts inside the block (profiling on: one stream), and under "all" every launch."""
    for kd in KINDS:
        smb.profile_read(kd, reset=True)
    got = {}
    smb.profile_enable(True)
    before = smb.launch_count()
    try:
        yield got
    finally:
        got["all"] = smb.launch_count() - before
        smb.profile_enable(False)
        for kd in KINDS:
            got[kd] = smb.profile_read(kd, reset=True)[1]


def sketch_launches(c):
    return sum(c[kd] for kd in KINDS)


def seqs_of(buf, offsets):
    return [buf[int(offsets[s]):int(offsets[s + 1])] for s in range(len(offsets) - 1)]


def templates(params):
    return [smb.KmerMinHash(num, k, prot, seed, mx, False) for num, k, prot, seed, mx in params]


def oracle_rows(p, buf, offsets, abund=False):
    num, k, prot, seed, mx = p
    return orc.sketch_each(buf, offsets, num, k, prot, seed, mx, abund, NT)


def survivors(p, buf, offsets, lens):
    """The call's survivor count for template p: every window whose hash is at or below the threshold, i.e. the summed
    abundances of oracle sketches with track_abundance at that threshold."""
    num, k, prot, seed, mx = p
    thr, _ = threshold(p, lens)
    return sum(int(o.abunds_np().sum()) for o in orc.sketch_each(buf, offsets, 0, k, prot, seed, thr, True, NT))


def assert_rows(coll, osk, what):
    rows = coll.rows_np()
    assert len(rows) == len(osk), what
    got_len = np.array([r.size for r in rows], dtype=np.int64)
    want = [o.mins_np() for o in osk]
    want_len = np.array([w.size for w in want], dtype=np.int64)
    if not np.array_equal(got_len, want_len):
        s = int(np.flatnonzero(got_len != want_len)[0])
        raise AssertionError((what, "row", s, int(got_len[s]), int(want_len[s])))
    if rows and not np.array_equal(np.concatenate(rows + [np.zeros(0, np.uint64)]),
                                   np.concatenate(want + [np.zeros(0, np.uint64)])):
        s = next(i for i, (r, w) in enumerate(zip(rows, want)) if not np.array_equal(r, w))
        raise AssertionError((what, "row", s, rows[s][:4], want[s][:4]))


def check_call(buf, offsets, params, osks, on_device=None, one_template=True):
    """The call, profiled and then unprofiled; every row against the oracle; the DNA rows also against the one-template
    call.  Returns the profiled launch counts."""
    def call():
        if on_device is None:
            return smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
        t, to = on_device
        return smb.SketchCollection.sketch_sequences_multi(t.data_ptr(), to.data_ptr(), templates(params), on_device=True,
                                                           n_seqs=len(offsets) - 1)
    with counted() as c:
        colls = call()
    for m in range(len(params)):
        assert_rows(colls[m], osks[m], ("profiled", m))
    colls = call()
    for m, p in enumerate(params):
        assert_rows(colls[m], osks[m], ("unprofiled", m))
        num, k, prot, seed, mx = p
        if one_template and not prot:
            one = smb.SketchCollection.sketch_sequences(buf, offsets, num, k, seed, mx)
            assert_rows(one, osks[m], ("one-template", m))
    return c


def seed_where(start, want, thr=MAX_HASH_1000):
    """The first seed from `start` at which every word in want[True] hashes at or below thr and every word in
    want[False] above it."""
    s = start
    while not (all(orc.hash_murmur(w, s) <= thr for w in want.get(True, ()))
               and all(orc.hash_murmur(w, s) > thr for w in want.get(False, ()))):
        s += 1
    return s


A21, A25, A31, A33, A51 = (b"A" * k for k in (21, 25, 31, 33, 51))
K10, F10 = b"K" * 10, b"F" * 10      # the poly-A stretch in protein k = 30: poly-K forward, poly-F on the reverse strand
POLY = [A21, A25, A31, A33, A51, K10, F10]
QUIET = 1000


@pytest.fixture(scope="module", autouse=True)
def _quiet_seed():
    """QUIET: a seed at which no poly-A word survives MAX_HASH_1000 * 16"""
    global QUIET
    QUIET = seed_where(1000, {False: POLY}, MAX_HASH_1000 * 16)


def random_part(length, seed):
    return dirty(random_dna(length, seed), seed + 1, n_bad=max(1, length // 2000))


def batch_of(parts):
    return b"".join(parts), offsets_of([len(s) for s in parts]), [len(s) for s in parts]


# ------------------------------------------------------------------------------------------------
# 1. the exact end of a survivor region: cap survivors fit, cap + 1 re-run exactly that template
# ------------------------------------------------------------------------------------------------
BOUNDARY = {
    # (templates, index at the boundary, its poly-A words that survive / must not)
    "fused_member": lambda s: ([(0, 21, False, s, MAX_HASH_1000), (0, 31, False, s, MAX_HASH_1000),
                                (0, 51, False, s, MAX_HASH_1000)], 1, {True: [A31], False: [A21, A51]}),
    "generic_k": lambda s: ([(0, 25, False, s, MAX_HASH_1000), (0, 21, False, QUIET, MAX_HASH_1000),
                             (0, 31, False, QUIET, MAX_HASH_1000), (0, 51, False, QUIET, MAX_HASH_1000)], 0,
                            {True: [A25]}),
    "protein": lambda s: ([(0, 30, True, s, MAX_HASH_1000), (0, 21, False, QUIET, MAX_HASH_1000),
                           (0, 31, False, QUIET, MAX_HASH_1000), (0, 51, False, QUIET, MAX_HASH_1000)], 0,
                          {True: [K10], False: [F10]}),
}


@pytest.mark.parametrize("kind", list(BOUNDARY))
def test_survivor_region_boundary(kind):
    seed = seed_where(0x5EED5000, BOUNDARY[kind](0)[2])
    params, b, _ = BOUNDARY[kind](seed)
    # the template right after the boundary one has survivors of its own from a launch that runs first (or, for the
    # fused member, early in the same launch): an entry written at index cap would land on its first entry
    assert params[b + 1][2] is False and params[b + 1][1] in (21, 51)
    head = [random_part(9000 + 1000 * i, 0x5EED5100 + i) for i in range(6)]
    p_b = params[b]
    base_lens = [len(s) for s in head]
    base_count = survivors(p_b, *batch_of(head)[:2], base_lens)

    def shape(run):
        parts = head + [polya_input(run, 1000, 0x5EED5200)]   # the poly-A sequence last: its survivors come last
        buf, offsets, lens = batch_of(parts)
        tail = survivors(p_b, parts[-1], [0, len(parts[-1])], [len(parts[-1])])
        return parts, buf, offsets, lens, base_count + tail - cap_of(p_b, lens)

    # tune the poly-A run one window at a time until the survivor count is exactly cap, then cap + 1
    guess = cap_of(p_b, base_lens) - base_count + (10 if p_b[2] else p_b[1])
    found = {}
    for run in range(guess - 40, guess + 80):
        d = shape(run)[-1]
        if d in (0, 1) and d not in found:
            found[d] = run
        if len(found) == 2:
            break
    assert set(found) == {0, 1}, (kind, guess)
    launches = {}
    for delta in (0, 1):
        parts, buf, offsets, lens, d = shape(found[delta])
        assert d == delta
        counts = [survivors(p, buf, offsets, lens) for p in params]
        caps = [cap_of(p, lens) for p in params]
        assert counts[b] == caps[b] + delta
        assert all(c <= cap for m, (c, cap) in enumerate(zip(counts, caps)) if m != b)
        assert counts[b + 1] > 0
        osks = [oracle_rows(p, buf, offsets) for p in params]
        c = check_call(buf, offsets, params, osks)
        launches[delta] = c
        assert c["sketch_multi"] == 1, c
        if kind == "fused_member":
            assert c["sketch_k31"] == delta and sketch_launches(c) == 1 + delta, c
        elif kind == "generic_k":
            assert c["sketch_other"] == 1 + delta and sketch_launches(c) == 1 + delta + 1, c
        else:
            assert sketch_launches(c) == 1, c
        # every launch of the call: one control-word reset per attempt, the sketch launches, the translation and a
        # hash per protein run, the grouping of each template
        prot_runs = (1 + delta) if kind == "protein" else 0
        want = (1 + delta) + sketch_launches(c) + (translate_launches(lens) if prot_runs else 0) + prot_runs \
            + sum(group_launches(cnt, len(lens), threshold(p, lens)[0]) for cnt, p in zip(counts, params))
        assert c["all"] == want, (c, want)
    # the shape of the two calls differs only by the re-run: group_survivors launches the same at cap and cap + 1
    if kind == "protein":
        assert launches[1]["all"] - launches[0]["all"] == 2


# ------------------------------------------------------------------------------------------------
# 2. re-run shapes in one call
# ------------------------------------------------------------------------------------------------
BIG = MAX_HASH_1000 * 16


def rerun_params(shape):
    """(templates, indices that overflow); the overflowing templates' poly-A words survive at their seeds"""
    s_gen = seed_where(0x5EED5300, {True: [A25]}, BIG)
    s_prot = seed_where(0x5EED5400, {True: [K10]}, BIG)
    if shape == "index_ge_1":
        return [(0, 21, False, QUIET, BIG), (0, 25, False, s_gen, BIG), (0, 31, False, QUIET, BIG),
                (0, 30, True, QUIET, BIG)], {1}
    if shape == "fused_21_51":
        s = seed_where(0x5EED5500, {True: [A21, A51], False: [A31]}, BIG)
        return [(0, 21, False, s, BIG), (0, 31, False, s, BIG), (0, 51, False, s, BIG), (0, 33, False, QUIET, BIG),
                (0, 30, True, QUIET, BIG)], {0, 2}
    if shape == "all":
        s = seed_where(0x5EED5600, {True: [A21, A31, A51]}, BIG)
        return [(0, 21, False, s, BIG), (0, 31, False, s, BIG), (0, 51, False, s, BIG), (0, 25, False, s_gen, BIG),
                (0, 30, True, s_prot, BIG)], {0, 1, 2, 3, 4}
    if shape == "protein_alone":
        return [(0, 21, False, QUIET, BIG), (0, 31, False, QUIET, BIG), (0, 51, False, QUIET, BIG),
                (0, 30, True, s_prot, BIG)], {3}
    assert shape == "protein_and_generic"
    return [(0, 21, False, QUIET, BIG), (0, 31, False, QUIET, BIG), (0, 25, False, s_gen, BIG), (0, 30, True, s_prot, BIG),
            (0, 51, False, QUIET, BIG), (0, 33, False, QUIET, BIG)], {2, 3}


@pytest.fixture(scope="module")
def rerun_batch():
    parts = [random_part(5000 + 700 * i, 0x5EED5700 + i) for i in range(12)]
    parts[4] = polya_input(30_000, 1000, 0x5EED5800)
    parts[9] = polya_input(25_000, 500, 0x5EED5801)
    parts[6] = b""
    return batch_of(parts)


# the sketch launches of each call: (multi, k21, k31, k51, other)
RERUN_LAUNCHES = {
    "index_ge_1": (1, 0, 0, 0, 2),          # 21+31 fused; 25 twice
    "fused_21_51": (2, 0, 0, 0, 1),         # 21+31+51 fused, then 21+51 fused again; 33 once
    "all": (2, 0, 0, 0, 2),                 # everything again, the fused trio as one launch
    "protein_alone": (1, 0, 0, 0, 0),
    "protein_and_generic": (1, 0, 0, 0, 3),  # 25 twice, 33 once
}


@pytest.mark.parametrize("shape", list(RERUN_LAUNCHES))
def test_rerun_shapes(shape, rerun_batch):
    buf, offsets, lens = rerun_batch
    params, over = rerun_params(shape)
    assert 4 <= len(params) <= MAX_TEMPLATES
    counts = [survivors(p, buf, offsets, lens) for p in params]
    caps = [cap_of(p, lens) for p in params]
    assert {m for m in range(len(params)) if counts[m] > caps[m]} == over, (counts, caps)
    assert all(c > 0 for c in counts)
    osks = [oracle_rows(p, buf, offsets) for p in params]
    c = check_call(buf, offsets, params, osks)
    assert (c["sketch_multi"], c["sketch_k21"], c["sketch_k31"], c["sketch_k51"], c["sketch_other"]) \
        == RERUN_LAUNCHES[shape], c
    n_prot = sum(1 for p in params if p[2])
    prot_runs = n_prot + sum(1 for m in over if params[m][2])
    want = 2 + sketch_launches(c) + translate_launches(lens) + prot_runs \
        + sum(group_launches(cnt, len(lens), threshold(p, lens)[0]) for cnt, p in zip(counts, params))
    assert c["all"] == want, (c, want)


# ------------------------------------------------------------------------------------------------
# 3. radix passes over sequence ids: 255, 256, 65 535 and 65 536 sequences
# ------------------------------------------------------------------------------------------------
def reads_batch(n_seqs, seed):
    """ragged reads of 60-150 bp with empty reads, reads shorter than k and dirty bytes"""
    r = splitmix64(seed, n_seqs + 8)
    lens = [int(60 + x % np.uint64(91)) for x in r[:n_seqs]]
    for i in range(0, n_seqs, 97):
        lens[i] = 0
    for i in range(13, n_seqs, 101):
        lens[i] = int(r[i] % np.uint64(21))
    offsets = offsets_of(lens)
    buf = dirty(random_dna(int(offsets[-1]), seed + 1), seed + 2, n_bad=max(8, n_seqs // 4))
    return buf, offsets, lens


SEQ_TEMPLATES = [(0, 21, False, 42, MAX_HASH_1000), (0, 31, False, 42, MAX_HASH_1000),
                 (0, 51, False, 42, MAX_HASH_1000), (0, 30, True, 42, MAX_HASH_1000 * 20), (1000, 21, False, 7, 0)]


@pytest.mark.parametrize("n_seqs, passes", [(255, 1), (256, 2), (65535, 2), (65536, 3)])
def test_sequence_id_sort_passes(n_seqs, passes):
    buf, offsets, lens = reads_batch(n_seqs, 0x5EED5900 + n_seqs)
    assert sort_passes(bits_of(n_seqs)) == passes
    # the hash sort: 7 passes at scaled = 1000 (odd: the result is copied back), 8 at scaled = 50 and keep-all
    assert [sort_passes(bits_of(threshold(p, lens)[0])) for p in SEQ_TEMPLATES] == [7, 7, 7, 8, 8]
    assert threshold(SEQ_TEMPLATES[4], lens)[0] == U64_MAX   # num = 1000 over reads: every window survives
    osks = [oracle_rows(p, buf, offsets) for p in SEQ_TEMPLATES]
    # survivors reach the last sequence ids
    for m in (3, 4):
        assert any(o.size() for o in osks[m][-64:])
    check_call(buf, offsets, SEQ_TEMPLATES, osks)


# ------------------------------------------------------------------------------------------------
# 4. survivor and slot counts past two levels of the scan and several grid-stride iterations
# ------------------------------------------------------------------------------------------------
def valid_windows(seq, k):
    a = np.frombuffer(seq.upper(), dtype=np.uint8)
    if a.size < k:
        return 0
    bad = ~np.isin(a, np.frombuffer(b"ACGT", dtype=np.uint8))
    c = np.concatenate([[0], np.cumsum(bad)])
    return int(np.count_nonzero(c[k:] == c[:-k]))


@pytest.fixture(scope="module")
def big_dna():
    """5.4 Mbp in 60 ragged sequences, one with a 40 kbp poly-A stretch"""
    r = splitmix64(0x5EED5A00, 64)
    parts = [random_part(int(40_000 + x % np.uint64(100_000)), 0x5EED5B00 + i) for i, x in enumerate(r[:60])]
    parts[17] = parts[17][:20_000] + b"A" * 40_000 + parts[17][20_000:]
    parts[33] = b""
    buf, offsets, lens = batch_of(parts)
    assert sum(lens) > 5_000_000
    return buf, offsets, lens


def test_keep_all_dna_past_two_scan_levels(big_dna):
    buf, offsets, lens = big_dna
    params = [(0, 21, False, 42, U64_MAX), (0, 31, False, 42, U64_MAX), (0, 51, False, 42, U64_MAX)]
    seqs = seqs_of(buf, offsets)
    for p in params:
        count = sum(valid_windows(s, p[1]) for s in seqs)
        assert count <= cap_of(p, lens)
        assert count > SCAN_TILE ** 2 and scan_levels(count) == 2       # the survivor scan recurses twice
        assert -(-count // MANY_THREADS) >= 7                           # grid-stride iterations of sketch_many.cu
        assert 256 * -(-count // RS_TILE) > SCAN_TILE                   # the sort's count-table scan recurses
        assert sort_passes(bits_of(U64_MAX)) == 8
    osks = [oracle_rows(p, buf, offsets) for p in params]
    c = check_call(buf, offsets, params, osks)
    assert c["sketch_multi"] == 1 and sketch_launches(c) == 1, c


def test_keep_all_protein_past_two_scan_levels():
    r = splitmix64(0x5EED5C00, 200)
    parts = [random_part(int(5000 + x % np.uint64(25_000)), 0x5EED5D00 + i) for i, x in enumerate(r[:150])]
    parts[40] = b""
    parts[41] = parts[41][:29]
    buf, offsets, lens = batch_of(parts)
    slots = 2 * sum(lens) + 6 * len(lens)
    assert slots > SCAN_TILE ** 2 and scan_levels(slots + 1) == 2
    assert -(-slots // PROTEIN_THREADS) >= 3
    params = [(0, 30, True, 42, U64_MAX), (0, 21, True, 9, U64_MAX)]
    osks = [oracle_rows(p, buf, offsets) for p in params]
    assert sum(o.size() for o in osks[0]) > 2 * MANY_THREADS
    check_call(buf, offsets, params, osks)


# ------------------------------------------------------------------------------------------------
# 5. more tiles than the persistent grid, several fast-path launches sharing one tile counter
# ------------------------------------------------------------------------------------------------
def test_persistent_grid_and_the_shared_tile_counter(big_dna):
    import torch
    buf, offsets, lens = big_dna
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    assert -(-sum(lens) // SK_TILE) > sm * SK_CTAS_PER_SM   # CTAs take tiles from the counter
    mx = MAX_HASH_1000 * 4
    s31 = seed_where(0x5EED5E00, {True: [A31]}, mx)
    q2 = seed_where(QUIET + 1, {False: POLY}, MAX_HASH_1000 * 16)
    cases = [
        # a fused pair plus a fast k at another seed: two fast launches
        ("fused_plus_fast", [(0, 21, False, QUIET, mx), (0, 51, False, QUIET, mx), (0, 31, False, q2, mx)], True,
         (1, 0, 1, 0, 0)),
        # fusion off: three fast launches
        ("fusion_off", [(0, 21, False, q2, mx), (0, 31, False, q2, mx), (0, 51, False, q2, mx)], False, (0, 1, 1, 1, 0)),
        # a fast-path re-run: k = 31 at its own seed, where the poly-A 31-mer survives, overflows and runs again
        ("fast_rerun", [(0, 21, False, QUIET, mx), (0, 31, False, s31, mx), (0, 51, False, QUIET, mx)], True,
         (1, 0, 2, 0, 0)),
    ]
    for name, params, fuse, want in cases:
        counts = [survivors(p, buf, offsets, lens) for p in params]
        over = [cnt > cap_of(p, lens) for cnt, p in zip(counts, params)]
        assert over == [False, name == "fast_rerun", False], (name, counts)
        osks = [oracle_rows(p, buf, offsets) for p in params]
        smb.fuse_multi_k(fuse)
        try:
            c = check_call(buf, offsets, params, osks)
        finally:
            smb.fuse_multi_k(True)
        assert (c["sketch_multi"], c["sketch_k21"], c["sketch_k31"], c["sketch_k51"], c["sketch_other"]) == want, (name, c)


# ------------------------------------------------------------------------------------------------
# 6. num sketches at scale: hundreds of rows cut short under the estimated threshold, sketched again on their own
# ------------------------------------------------------------------------------------------------
def test_num_estimates_redo_hundreds_of_rows():
    import torch
    r = splitmix64(0x5EED5F00, 4000)
    lens = [int(x % np.uint64(130)) if i % 9 == 0 else int(300 + x % np.uint64(4000)) for i, x in enumerate(r[:3000])]
    offsets = offsets_of(lens)
    buf = dirty(random_dna(int(offsets[-1]), 0x5EED5F01), 0x5EED5F02, n_bad=3000)
    params = [(100, 21, False, 42, 0), (100, 30, True, 5, 0), (0, 31, False, 42, MAX_HASH_1000 * 8)]
    for p in params[:2]:
        thr, frac = threshold(p, lens)
        assert frac < 1.0
        short = [o.size() < p[0] for o in oracle_rows((0, p[1], p[2], p[3], thr), buf, offsets)]
        assert 200 <= sum(short) < len(lens) // 2, sum(short)
    osks = [oracle_rows(p, buf, offsets) for p in params]
    check_call(buf, offsets, params, osks)
    t = torch.frombuffer(bytearray(buf + b"\0" * (-len(buf) % 16)), dtype=torch.uint8).cuda()
    to = torch.from_numpy(offsets.view(np.int64)).cuda()
    check_call(buf, offsets, params, osks, on_device=(t, to))


# ------------------------------------------------------------------------------------------------
# 7. empty results
# ------------------------------------------------------------------------------------------------
def assert_compare(coll, osk):
    got = smb.compare_matrix(coll, coll)
    oc, osz = orc.compare_matrix(osk, osk, NT)
    assert np.array_equal(got[0], oc) and np.array_equal(got[1], osz)


def test_empty_templates_next_to_full_ones():
    r = splitmix64(0x5EED6000, 64)
    lens = [int(100 + x % np.uint64(4000)) for x in r[:40]] + [0, 3, 30]
    offsets = offsets_of(lens)
    buf = dirty(random_dna(int(offsets[-1]), 0x5EED6001), 0x5EED6002, n_bad=40)
    long_k = max(lens) + 1
    params = [(0, 21, False, 42, 1), (0, 31, False, 42, MAX_HASH_1000 * 20), (0, long_k, False, 42, U64_MAX),
              (0, 3 * (max(lens) // 3 + 1), True, 42, U64_MAX), (0, 30, True, 42, MAX_HASH_1000 * 20),
              (0, 51, False, 42, U64_MAX)]
    counts = [survivors(p, buf, offsets, lens) for p in params]
    assert counts[0] == counts[2] == counts[3] == 0 and min(counts[1], counts[4]) > 1000 and counts[5] > 50_000
    osks = [oracle_rows(p, buf, offsets) for p in params]
    check_call(buf, offsets, params, osks)
    colls = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    for coll, osk in zip(colls, osks):
        assert_compare(coll, osk)


def test_three_hundred_empty_sequences():
    offsets = np.zeros(301, dtype=np.uint64)
    params = [(0, 21, False, 42, MAX_HASH_1000), (0, 31, False, 42, MAX_HASH_1000), (0, 51, False, 42, MAX_HASH_1000),
              (0, 30, True, 42, MAX_HASH_1000), (50, 25, False, 42, 0)]
    osks = [oracle_rows(p, b"", offsets) for p in params]
    assert all(o.size() == 0 for osk in osks for o in osk)
    c = check_call(b"", offsets, params, osks)
    assert sketch_launches(c) == 0, c
    colls = smb.SketchCollection.sketch_sequences_multi(b"", offsets, templates(params))
    for coll, osk in zip(colls, osks):
        assert len(coll) == 300
        assert_compare(coll, osk)


# ------------------------------------------------------------------------------------------------
# 8. one context, calls of changing shape: stale scratch sizes, tile counters re-armed between calls
# ------------------------------------------------------------------------------------------------
def test_calls_of_changing_shape_on_one_context(big_dna):
    import torch
    buf, offsets, lens = big_dna
    mx = MAX_HASH_1000 * 4
    large = [(0, 21, False, 42, mx), (0, 31, False, 42, mx), (0, 51, False, 42, mx), (0, 30, True, 42, mx)]
    check_call(buf, offsets, large, [oracle_rows(p, buf, offsets) for p in large], one_template=False)
    sbuf, soff, slens = reads_batch(300, 0x5EED6100)
    small = [(0, 31, False, 3, MAX_HASH_1000 * 50), (200, 21, False, 42, 0)]
    check_call(sbuf, soff, small, [oracle_rows(p, sbuf, soff) for p in small], one_template=False)
    # the per-object path on the same context
    gs = [smb.KmerMinHash(0, 21, False, 42, mx, True), smb.KmerMinHash(500, 51, False, 42, 0, False)]
    smb.add_sequences(gs, buf[:2_000_000], [0, 700_000, 2_000_000])
    for g, (num, k, mxx) in zip(gs, ((0, 21, mx), (500, 51, 0))):
        o = orc.KmerMinHash(num, k, False, 42, mxx, num == 0)
        o.add_sequence(buf[:700_000], True)
        o.add_sequence(buf[700_000:2_000_000], True)
        assert np.array_equal(g.mins_np(), o.mins_np())
    # a large call with other templates, from device memory
    other = [(0, 25, False, 11, mx), (0, 21, False, 11, mx), (0, 51, False, 11, mx), (0, 24, True, 11, mx),
             (0, 31, False, 12, mx), (2000, 31, False, 42, 0)]
    t = torch.frombuffer(bytearray(buf + b"\0" * (-len(buf) % 16)), dtype=torch.uint8).cuda()
    to = torch.from_numpy(offsets.view(np.int64)).cuda()
    check_call(buf, offsets, other, [oracle_rows(p, buf, offsets) for p in other], on_device=(t, to))
