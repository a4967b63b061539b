"""The sketch path at the boundaries its kernels and host loop special-case, bit for bit against the oracle.

- seeds other than 42 through every device hash (fast kernels alone and fused, the generic kernel, protein,
  smgpu_sketch_collection) and the host hash;
- every DNA k from 1 to 96, long k up to SK_MAX_GENERIC_K = 8192 (halo wider than a tile past k = 4097) and the
  refusal above it; protein k from 3 to 99 and a few long ones;
- host batches larger than a chunk of the overlapped host-to-device copy (more chunk edges, at 1 MiB chunks, in
  tests/workers/sketch_chunk_worker.py);
- the re-run loops of add_sequences (candidate overflow, estimate widening, the lazy fold of a scaled sketch past
  2^22 candidates) and the survivor-overflow loop of smgpu_sketch_collection, reached on purpose with a poly-A
  stretch whose k-mer hashes below the threshold;
- batch shape: 6 sketches per call, 7 refused, a sketch twice in one call refused, device-resident ragged batches.

A test that exists to reach a branch asserts that it did, from a shape fact computed from the constants below or
from the launch counts of the per-kernel profiler, so that a changed constant fails the test instead of silently
skipping the branch.  Profiling keeps every kernel on one stream, so multi-sketch cases run once profiled (to count
launches) and once unprofiled (each sketch on its own stream); both must equal the oracle."""
import contextlib
import os
import re

import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from util import MAX_HASH_1000, make_reads, random_dna, splitmix64

pytestmark = pytest.mark.gpu

SK_TILE = 4096                 # window starts per tile (kernels.cuh)
SK_MAX_GENERIC_K = 8192        # largest k the device sketcher takes (kernels.cuh)
H2D_CHUNK = 8 << 20            # default chunk of the host-to-device copy (minhash.cu, SMB200_H2D_CHUNK_MB)
LAZY_CANDIDATES = 1 << 22      # a scaled sketch folds its candidates in past this many (minhash.cu)
MAX_SKETCHES = 6               # sketches per batch call (include/sourmash_b200.h)
ERR_INTERNAL = 2
SEEDS = [0, 1, 2**32 - 1, 2**32, 2**63, 2**64 - 1]
KINDS = ("sketch_k21", "sketch_k31", "sketch_k51", "sketch_other", "sketch_multi")


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


# ------------------------------------------------------------------------------------------------
# helpers (also used by tests/workers/sketch_chunk_worker.py)
# ------------------------------------------------------------------------------------------------
def pair(num, k, max_hash=0, abund=False, seed=42, protein=False):
    return (smb.KmerMinHash(num, k, protein, seed, max_hash, abund),
            orc.KmerMinHash(num, k, protein, seed, max_hash, abund))


def same(g, o):
    assert np.array_equal(g.mins_np(), o.mins_np()), (g.mins_np()[:5], o.mins_np()[:5], g.size(), o.size())
    ga, oa = g.abunds_np(), o.abunds_np()
    assert (ga is None) == (oa is None)
    if ga is not None:
        assert np.array_equal(ga, oa)
    assert g.md5sum() == o.md5sum()


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


def offsets_of(lens):
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)


def oracle_batch(os_, buf, offsets, force):
    """The batch call on the oracle: for every sketch, its sequences in order, stopping at its first invalid k-mer.
    Returns the message of the first sketch (in call order) that failed, or None."""
    first = None
    for o in os_:
        for s in range(len(offsets) - 1):
            try:
                o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], force)
            except orc.SourmashError as e:
                assert e.code == 1101
                first = first or e.message
                break
    return first


def gpu_batch(gs, buf, offsets, force):
    """smb.add_sequences; returns the error message or None"""
    try:
        smb.add_sequences(gs, buf, offsets, force=force)
    except smb.SourmashError as e:
        assert e.code == 1101, e
        return e.message
    return None


def tiles_ready(k, n_bytes):
    """sketch_tiles_ready (sketch.cu): tiles whose window starts and halo lie in the first n_bytes"""
    b = SK_TILE + (k - 1 + 15) // 16 * 16
    return 0 if n_bytes < b else (n_bytes - b) // SK_TILE + 1


def chunk_ends(n, chunk, packed_read_len=0):
    """Bytes on the device after each host-to-device copy of add_sequences (minhash.cu) for a host batch of n bytes;
    packed_read_len for 2-bit reads, whose chunks hold whole reads."""
    ends, copied, c = [], 0, chunk
    while True:
        left = n - copied
        ln = min(c, left)
        if left > (2 << 20):
            ln = min(ln, max((left // 2 + 4095) & ~4095, 2 << 20))
        c = min(c * 2, chunk)
        if packed_read_len:
            r0 = copied // packed_read_len
            r1 = min(n // packed_read_len, max(r0 + 1, (copied + ln) // packed_read_len))
            ln = r1 * packed_read_len - copied
        copied += ln
        ends.append(copied)
        if copied >= n:
            return ends


def sketch_launches(k, ends):
    """Sketch launches of one k (a fused group: its widest k) over the chunks that land at `ends`."""
    n = ends[-1]
    total = (n + SK_TILE - 1) // SK_TILE
    lo = count = 0
    for e in ends:
        hi = total if e >= n else min(total, tiles_ready(k, e))
        if hi > lo:
            count += 1
            lo = hi
    return count


@contextlib.contextmanager
def counted():
    """Per-kernel launch counts of the sketch kernels inside the block (profiling on: one stream)."""
    for kd in KINDS:
        smb.profile_read(kd, reset=True)
    got = {}
    smb.profile_enable(True)
    try:
        yield got
    finally:
        smb.profile_enable(False)
        for kd in KINDS:
            got[kd] = smb.profile_read(kd, reset=True)[1]


def kind_of(k):
    return {21: "sketch_k21", 31: "sketch_k31", 51: "sketch_k51"}.get(k, "sketch_other")


def polya_seed(k, start):
    """The first seed from `start` at which the canonical poly-A k-mer hashes at or below MAX_HASH_1000."""
    s = start
    while orc.hash_murmur(b"A" * k, s) > MAX_HASH_1000:
        s += 1
    return s


def polya_run(seq, k):
    """windows of seq whose canonical k-mer is poly-A (the one long A-run of seq; flanks are random)"""
    return max(len(m) for m in re.findall(rb"A+", seq)) - k + 1


def polya_input(n_polya, flank, seed):
    left, right = random_dna(flank, seed), random_dna(flank, seed + 1)
    return left + b"A" * n_polya + right


# ------------------------------------------------------------------------------------------------
# 1. seeds
# ------------------------------------------------------------------------------------------------
SEED_LENS = [9000, 0, 20, 21, 51, 300, 4200, 52, 7000, 13]


@pytest.mark.parametrize("seed", SEEDS)
def test_seeds_through_every_sketch_kernel(seed):
    offsets = offsets_of(SEED_LENS)
    buf = dirty(random_dna(int(offsets[-1]), 0x5EED0100), 0x5EED0101)
    mx = MAX_HASH_1000 * 50
    for k in (21, 31, 51, 9, 16, 33, 70):
        g, o = pair(0, k, mx, True, seed)
        with counted() as n:
            smb.add_sequences([g], buf, offsets)
        assert n[kind_of(k)] == 1 and sum(n.values()) == 1
        oracle_batch([o], buf, offsets, True)
        same(g, o)
    # fused 21/31/51 at this seed: one launch serves the three
    kinds = ((0, mx, True), (500, 0, False), (200, 0, True))
    for profiled in (True, False):
        gos = [pair(num, k, m, ab, seed) for k, (num, m, ab) in zip((21, 31, 51), kinds)]
        if profiled:
            with counted() as n:
                smb.add_sequences([g for g, _ in gos], buf, offsets)
            assert n["sketch_multi"] == 1 and sum(n.values()) == 1
        else:
            smb.add_sequences([g for g, _ in gos], buf, offsets)
        oracle_batch([o for _, o in gos], buf, offsets, True)
        for g, o in gos:
            same(g, o)
    for k in (21, 48):
        g, o = pair(0, k, mx, True, seed, protein=True)
        smb.add_sequences([g], buf, offsets)
        oracle_batch([o], buf, offsets, True)
        same(g, o)
    for num, m in ((300, 0), (0, mx)):
        rows = smb.SketchCollection.sketch_sequences(buf, offsets, num, 31, seed, m).rows_np()
        for s in range(len(SEED_LENS)):
            o = orc.KmerMinHash(num, 31, False, seed, m, False)
            o.add_sequence(buf[int(offsets[s]):int(offsets[s + 1])], True)
            assert np.array_equal(rows[s], o.mins_np()), s


@pytest.mark.parametrize("seed", SEEDS)
def test_seeds_host_hash_and_add_word(seed):
    r = splitmix64(seed ^ 0x77, 64)
    words = [b"", b"A", b"acgt"] + [random_dna(int(1 + x % np.uint64(70)), int(x)) for x in r[:40]] + [random_dna(300, 3)]
    g, o = pair(0, 5, 2**63, True, seed)
    for w in words:
        assert smb.hash_murmur(w, seed) == orc.hash_murmur(w, seed), w
        g.add_word(w); o.add_word(w)
    same(g, o)


def test_mixed_seed_batch_fuses_only_the_matching_seed():
    offsets = offsets_of(SEED_LENS)
    buf = dirty(random_dna(int(offsets[-1]), 0x5EED0102), 0x5EED0103)
    spec = ((21, 42), (31, 42), (51, 7))
    for profiled in (True, False):
        gos = [pair(0, k, MAX_HASH_1000 * 50, True, s) for k, s in spec]
        gs = [g for g, _ in gos]
        if profiled:
            with counted() as n:
                smb.add_sequences(gs, buf, offsets)
            # the pair at seed 42 shares a launch, the sketch at seed 7 has its own
            assert n["sketch_multi"] == 1 and n["sketch_k51"] == 1 and sum(n.values()) == 2
        else:
            smb.add_sequences(gs, buf, offsets)
        oracle_batch([o for _, o in gos], buf, offsets, True)
        for g, o in gos:
            same(g, o)


def test_compare_and_merge_across_seeds_refused():
    seq = random_dna(5000, 0x5EED0104)
    for s0, s1 in ((42, 7), (0, 2**64 - 1), (2**32, 2**32 - 1)):
        (a, oa), (b, ob) = pair(100, 21, 0, False, s0), pair(100, 21, 0, False, s1)
        for x in (a, oa, b, ob):
            x.add_sequence(seq, True)
        for op in ("compare", "merge", "count_common"):
            with pytest.raises(smb.SourmashError) as ge:
                getattr(a, op)(b)
            with pytest.raises(orc.SourmashError) as oe:
                getattr(oa, op)(ob)
            assert ge.value.code == oe.value.code == 104
            assert ge.value.message == oe.value.message == "mismatch in seed; comparison fail"
        same(a, oa)


# ------------------------------------------------------------------------------------------------
# 2. k: every DNA k to 96, long k, the refusal above SK_MAX_GENERIC_K; protein k
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", range(1, 97))
def test_every_dna_k_to_96(k):
    n = 2 * SK_TILE + (k * 997) % SK_TILE     # two to three tiles
    seq = dirty(random_dna(n, 0x5EED0200 + k), 0x5EED0300 + k, n_bad=8)
    g, o = pair(0, k, 2**63, True)
    smb.add_sequences([g], seq, [0, n])
    o.add_sequence(seq, True)
    if k >= 8:   # (below, the few canonical k-mers may all hash above max_hash)
        assert o.size() > 1000
    same(g, o)
    # a second sequence on top of the state: repeats raise abundances
    seq2 = seq[1000:4000] + random_dna(700, k)
    g.add_sequence(seq2, True); o.add_sequence(seq2, True)
    same(g, o)


LONG_K = [127, 128, 129, 255, 256, 1000, 4095, 4096, 4097, 8191, 8192]


@pytest.mark.parametrize("k", LONG_K)
def test_long_k_around_whole_tiles(k):
    assert k <= SK_MAX_GENERIC_K
    for m in (1, 2):
        for n in (SK_TILE * m + k - 2, SK_TILE * m + k - 1, SK_TILE * m + k):
            a = bytearray(random_dna(n, 0x5EED0400 + k + n))
            bad = [3, n - 5] if m == 1 else [3, n // 2, n - 5]
            for p in bad:                       # the long-k bitmap loop marks the windows around each
                a[p] = ord("N")
            a[n // 3:n // 3 + 40] = bytes(a[n // 3:n // 3 + 40]).lower()
            seq = bytes(a)
            g, o = pair(0, k, 2**63, True)
            smb.add_sequences([g], seq, [0, n])
            o.add_sequence(seq, True)
            same(g, o)
    if k > SK_TILE + 1:   # the halo alone is wider than a tile
        assert SK_TILE + (k - 1 + 15) // 16 * 16 > 2 * SK_TILE


@pytest.mark.parametrize("k", [127, 1000, 4097, 8192])
def test_long_k_force_false_stops_where_the_oracle_stops(k):
    n = 2 * SK_TILE + k - 1
    a = bytearray(random_dna(n, 0x5EED0500 + k))
    a[k + SK_TILE + 100] = ord("N")   # the first failing window starts in the second tile
    seq = bytes(a)
    g, o = pair(0, k, 2**63, True)
    with pytest.raises(smb.SourmashError) as ge:
        g.add_sequence(seq, False)
    with pytest.raises(orc.SourmashError) as oe:
        o.add_sequence(seq, False)
    assert ge.value.code == oe.value.code == 1101
    assert ge.value.message == oe.value.message
    assert o.size() > 1000   # windows before the failing one were kept
    same(g, o)


def test_k_above_the_generic_limit_is_refused():
    k = SK_MAX_GENERIC_K + 1
    seq = random_dna(SK_TILE + k, 0x5EED0600)
    g = smb.KmerMinHash(0, k, False, 42, 2**63, True)
    with pytest.raises(smb.SourmashError) as e:
        smb.add_sequences([g], seq, [0, len(seq)])
    assert e.value.code == ERR_INTERNAL and "ksize above 8192" in e.value.message
    assert g.size() == 0
    # the context is still usable
    g2, o2 = pair(0, 21, 2**63, True)
    smb.add_sequences([g2], seq[:9000], [0, 9000])
    o2.add_sequence(seq[:9000], True)
    same(g2, o2)


@pytest.mark.parametrize("k", list(range(3, 100)) + [150, 300, 3003])
def test_protein_k(k):
    n = 3 * k + 2000
    seq = dirty(random_dna(n, 0x5EED0700 + k), 0x5EED0800 + k, n_bad=10)
    g, o = pair(0, k, 2**63, True, protein=True)
    smb.add_sequences([g], seq, [0, n])
    o.add_sequence(seq, True)
    assert o.size() > 0
    same(g, o)


# ------------------------------------------------------------------------------------------------
# 3. a host batch of many default-size chunks (1 MiB chunks: tests/workers/sketch_chunk_worker.py)
# ------------------------------------------------------------------------------------------------
def test_host_batch_of_24_mib_at_the_default_chunk_size():
    read_len = 151
    n_reads = (24 << 20) // read_len + 1
    reads = make_reads(random_dna(2_000_000, 0x5EED0900), n_reads, read_len, 0x5EED0901)
    n = n_reads * read_len
    ends = chunk_ends(n, H2D_CHUNK)
    assert len(ends) >= 4
    ks = [21, 31, 51]
    os_ = orc.mt_sketch_reads(reads, n_reads, read_len, ks, 0, MAX_HASH_1000, True, os.cpu_count() or 4)
    for profiled in (True, False):
        gs = [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000, True) for k in ks]
        if profiled:
            with counted() as c:
                smb.add_reads(gs, reads, n_reads, read_len, force=False)
            assert c["sketch_multi"] == sketch_launches(51, ends) == len(ends) and sum(c.values()) == len(ends)
        else:
            smb.add_reads(gs, reads, n_reads, read_len, force=False)
        for g, o in zip(gs, os_):
            same(g, o)


def test_chunked_batches_in_a_worker(tmp_path):
    import subprocess
    import sys
    worker = os.path.join(os.path.dirname(os.path.abspath(__file__)), "workers", "sketch_chunk_worker.py")
    env = dict(os.environ, SMB200_H2D_CHUNK_MB="1")
    p = subprocess.Popen([sys.executable, worker], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        out, _ = p.communicate(timeout=900)
    except subprocess.TimeoutExpired:
        p.kill()
        raise
    assert p.returncode == 0 and out.rstrip().endswith("ok"), out[-4000:]


# ------------------------------------------------------------------------------------------------
# 4. re-run paths, reached with a poly-A stretch whose k-mer survives the threshold
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [21, 31, 51, 33])
def test_candidate_overflow_and_estimate_widening(k):
    seed = polya_seed(k, 2**32 + 1000003 * k)
    seq = polya_input(300_000, 3000, 0x5EED0A00 + k)
    n = len(seq)
    h = orc.hash_murmur(b"A" * k, seed)
    windows = polya_run(seq, k)
    chunks = sketch_launches(k, chunk_ends(n, H2D_CHUNK))
    # scaled: every poly-A window survives, more than the candidate reservation holds -> one re-run
    assert windows > MAX_HASH_1000 / 2**64 * 1.25 * n + 4096
    g, o = pair(0, k, MAX_HASH_1000, True, seed)
    with counted() as c:
        smb.add_sequences([g], seq, [0, n])
    assert c[kind_of(k)] == chunks + 1 and sum(c.values()) == chunks + 1
    o.add_sequence(seq, True)
    same(g, o)
    i = int(np.searchsorted(g.mins_np(), np.uint64(h)))
    assert g.mins_np()[i] == h and g.abunds_np()[i] == windows
    # num + abundance: the estimated threshold keeps too few distinct hashes -> widened, after the overflow re-run
    num = 500
    want = 8.0 * num + 4096.0
    assert n > 4 * want and want / n > 2.0**-6   # the estimate is used, and one widening reaches the whole hash range
    est = int(want / n * 2**64)
    o_est = orc.KmerMinHash(0, k, False, seed, est, False)
    o_est.add_sequence(seq, True)
    assert o_est.size() < num and windows > want / n * 1.25 * n + 4096
    g, o = pair(num, k, 0, True, seed)
    with counted() as c:
        smb.add_sequences([g], seq, [0, n])
    assert c[kind_of(k)] == chunks + 2 and sum(c.values()) == chunks + 2
    o.add_sequence(seq, True)
    same(g, o)
    # unprofiled, and a second call on the state
    g, o = pair(num, k, 0, True, seed)
    for s in (seq, seq[:150_000] + random_dna(4000, k)):
        smb.add_sequences([g], s, [0, len(s)])
        o.add_sequence(s, True)
        same(g, o)


def test_lazy_fold_past_2_pow_22_candidates():
    k = 21
    seed = polya_seed(k, 2**63 + 12345)
    seq = polya_input(LAZY_CANDIDATES + 120_000, 2000, 0x5EED0B00)
    n = len(seq)
    windows = polya_run(seq, k)
    assert windows > LAZY_CANDIDATES
    ends = chunk_ends(n, H2D_CHUNK)
    g, o = pair(0, k, MAX_HASH_1000, True, seed)
    with counted() as c:
        smb.add_sequences([g], seq, [0, n])
    assert c["sketch_k21"] == sketch_launches(k, ends) + 1   # + the overflow re-run
    o.add_sequence(seq, True)
    same(g, o)
    # a second call lands on the folded state
    seq2 = random_dna(50_000, 0x5EED0B01) + b"A" * 100_000
    smb.add_sequences([g], seq2, [0, len(seq2)])
    o.add_sequence(seq2, True)
    same(g, o)
    h = orc.hash_murmur(b"A" * k, seed)
    i = int(np.searchsorted(g.mins_np(), np.uint64(h)))
    assert g.mins_np()[i] == h and g.abunds_np()[i] == windows + polya_run(seq2, k)


@pytest.mark.parametrize("num, mx", [(0, MAX_HASH_1000), (50, 0)])
def test_sketch_collection_survivor_overflow(num, mx):
    k = 21
    seed = polya_seed(k, 99991)
    lens, parts = [], []
    for i in range(15):
        if i % 5 == 2:
            s = polya_input(40_000, 1000, 0x5EED0C00 + i)
        else:
            s = dirty(random_dna(3000, 0x5EED0D00 + i), i)
        parts.append(s)
        lens.append(len(s))
    buf = b"".join(parts)
    offsets = offsets_of(lens)
    n = len(buf)
    # the survivor reservation of sketch_collection.cu, and what survives
    if mx:
        frac = mx / 2**64
    else:
        frac = min(1.0, 16.0 * num / float(np.median(lens)))
    survivors = sum(polya_run(s, k) for s in parts if b"A" * 1000 in s)
    assert survivors > frac * 1.25 * n + 4096
    if num:   # every row keeps num hashes under the estimated threshold: no row is sketched again on its own
        for s in parts:
            o = orc.KmerMinHash(0, k, False, seed, int(frac * 2**64), False)
            o.add_sequence(s, True)
            assert o.size() >= num
    with counted() as c:
        coll = smb.SketchCollection.sketch_sequences(buf, offsets, num, k, seed, mx)
    assert c["sketch_k21"] == 2 and sum(c.values()) == 2
    rows = coll.rows_np()
    for s in range(len(lens)):
        o = orc.KmerMinHash(num, k, False, seed, mx, False)
        o.add_sequence(parts[s], True)
        assert np.array_equal(rows[s], o.mins_np()), s


# ------------------------------------------------------------------------------------------------
# 5. batch shape
# ------------------------------------------------------------------------------------------------
def six_sketches(seed2=7):
    """fused 21/31/51 in mixed modes, generic 33, protein 30, and 31 at another seed"""
    mx = MAX_HASH_1000 * 20
    return [pair(0, 21, mx, True), pair(500, 31, 0, False), pair(300, 51, 0, True), pair(0, 33, mx, False),
            pair(0, 30, mx, True, protein=True), pair(0, 31, mx, True, seed2)]


def test_six_sketches_pass_and_seven_are_refused():
    r = splitmix64(0x5EED0E00, 64)
    lens = [int(x % np.uint64(3000)) for x in r[:40]]
    offsets = offsets_of(lens)
    buf = dirty(random_dna(int(offsets[-1]), 0x5EED0E01), 0x5EED0E02)
    gos = six_sketches()
    assert len(gos) == MAX_SKETCHES
    smb.add_sequences([g for g, _ in gos], buf, offsets)
    oracle_batch([o for _, o in gos], buf, offsets, True)
    for g, o in gos:
        same(g, o)
    seven = [g for g, _ in six_sketches()] + [smb.KmerMinHash(0, 21, False, 42, MAX_HASH_1000, True)]
    with pytest.raises(smb.SourmashError) as e:
        smb.add_sequences(seven, buf, offsets)
    assert e.value.code == ERR_INTERNAL and "at most 6 sketches" in e.value.message
    assert all(g.size() == 0 for g in seven)


@pytest.mark.parametrize("mode", ["scaled", "num_abund"])
@pytest.mark.parametrize("n", [2_000, 400_000])
@pytest.mark.parametrize("layout", ["gg", "ghg"])
def test_a_sketch_twice_in_one_call_is_refused(mode, n, layout):
    num, mx = (0, MAX_HASH_1000 * 50) if mode == "scaled" else (200, 0)
    want = 8.0 * num + 4096.0
    frac = mx / 2**64 if mx else (want / n if n > 4 * want else 1.0)
    # the large batch is above the candidate reservation of one pass: two passes over one sketch would not fit
    assert (2 * frac * n > frac * 1.25 * n + 4096) == (n > 100_000)
    first = random_dna(20_000, 0x5EED0F00)
    buf = random_dna(n, 0x5EED0F01 + n)
    g, og = pair(num, 21, mx, mode != "scaled")
    h, oh = pair(num, 31, mx, mode != "scaled")
    for x, y in ((g, og), (h, oh)):
        smb.add_sequences([x], first, [0, len(first)])
        y.add_sequence(first, True)
    mhs = [g, g] if layout == "gg" else [g, h, g]
    with pytest.raises(smb.SourmashError) as e:
        smb.add_sequences(mhs, buf, [0, n])
    assert e.value.code == ERR_INTERNAL and "more than once" in e.value.message
    same(g, og); same(h, oh)   # nothing was added
    for x, y in ((g, og), (h, oh)):
        smb.add_sequences([x], buf, [0, n])
        y.add_sequence(buf, True)
        same(x, y)
    smb.add_sequences([g, h], buf, [0, n])
    og.add_sequence(buf, True); oh.add_sequence(buf, True)
    same(g, og); same(h, oh)


def test_device_resident_ragged_batch():
    import torch
    r = splitmix64(0x5EED1000, 200)
    lens = [int(x % np.uint64(2500)) for x in r[:120]] + [0, 20, 21, 51, 30, 3]
    lens[-1] += (7 - sum(lens)) % 16   # total length 7 (mod 16): the tail is not a whole 16-byte group
    offsets = offsets_of(lens)
    n = int(offsets[-1])
    assert n % 16 == 7
    buf = dirty(random_dna(n, 0x5EED1001), 0x5EED1002, n_bad=30)
    # padded as the header requires: readable up to offsets[n_seqs] rounded up to 16
    t = torch.frombuffer(bytearray(buf + b"\0" * (-n % 16)), dtype=torch.uint8).cuda()
    assert t.numel() == (n + 15) // 16 * 16
    to = torch.from_numpy(offsets.view(np.int64)).cuda()
    mx = MAX_HASH_1000 * 50
    gos = [pair(0, 21, mx, True), pair(300, 31, 0, False), pair(0, 33, mx, True), pair(0, 30, mx, True, protein=True)]
    smb.add_sequences([g for g, _ in gos], t.data_ptr(), to.data_ptr(), on_device=True, n_seqs=len(lens))
    oracle_batch([o for _, o in gos], buf, offsets, True)
    for g, o in gos:
        same(g, o)
    # force=False on the device copy: the first invalid k-mer, as on the host
    gos = [pair(0, 21, mx, True), pair(0, 33, mx, True)]
    with pytest.raises(smb.SourmashError) as ge:
        smb.add_sequences([g for g, _ in gos], t.data_ptr(), to.data_ptr(), force=False, on_device=True, n_seqs=len(lens))
    assert ge.value.message == oracle_batch([o for _, o in gos], buf, offsets, False)
    for g, o in gos:
        same(g, o)
