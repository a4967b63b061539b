"""smgpu_sketch_collections: one collection per template, each row bit for bit the oracle loop
    for s in sequences: for t in templates: mh = KmerMinHash(t); mh.add_sequence(s, True); rows[t].append(mh.mins)
over ragged, dirty batches; fused and single-k launches, the shared protein translation, device-resident input,
the survivor overflow of one template in a multi-template call, and the refused template sets."""
import contextlib
import ctypes as C
import re

import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from util import MAX_HASH_1000, random_dna, splitmix64

pytestmark = pytest.mark.gpu

KINDS = ("sketch_k21", "sketch_k31", "sketch_k51", "sketch_other", "sketch_multi")
SCALED = MAX_HASH_1000 * 20
ERR_PANIC, ERR_INTERNAL, ERR_MISMATCH_DNAPROT = 1, 2, 102


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def dirty(seq: bytes, seed, n_bad=12):
    """sprinkle lower-case stretches and invalid bytes"""
    a = bytearray(seq)
    r = splitmix64(seed, n_bad * 2 + 8)
    for i in range(4):
        s = int(r[i] % np.uint64(max(1, len(a) - 50)))
        a[s:s + 40] = bytes(a[s:s + 40]).lower()
    for i in range(n_bad):
        a[int(r[8 + i] % np.uint64(len(a)))] = b"NRYn-*"[int(r[8 + n_bad + i] % np.uint64(6))]
    return bytes(a)


def offsets_of(lens):
    return np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)


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


def ragged_batch(seed):
    """Median ~24 kbp; empty sequences, sequences shorter than / exactly as long as each k used below (DNA 21, 25,
    31, 51; protein 24, 30, 31: 30 bytes hold ten codons, a whole window of protein k = 31, which the reference
    still skips), a few far shorter than the median (the num estimate cuts them short), dirty bytes, two sequences
    sharing most of their content and a repeated motif."""
    r = splitmix64(seed, 64)
    lens = [int(20000 + x % np.uint64(9000)) for x in r[:14]] + [0, 20, 21, 24, 25, 30, 31, 51, 7, 300, 2500, 0, 60000]
    offsets = offsets_of(lens)
    buf = dirty(random_dna(int(offsets[-1]), seed + 1), seed + 2, n_bad=40)
    a, b = int(offsets[1]), int(offsets[2])
    buf = buf[:a] + buf[:b - a] + buf[b:]
    m0 = int(offsets[5])
    buf = buf[:m0] + (b"ACGTTGCA" * 4000)[:lens[5]] + buf[m0 + lens[5]:]
    return buf, offsets


def seqs_of(buf, offsets):
    return [buf[int(offsets[s]):int(offsets[s + 1])] for s in range(len(offsets) - 1)]


def templates(params):
    return [smb.KmerMinHash(num, k, prot, seed, mx, False) for num, k, prot, seed, mx in params]


def oracle_sketches(p, seqs):
    num, k, prot, seed, mx = p
    out = []
    for s in seqs:
        o = orc.KmerMinHash(num, k, prot, seed, mx, False)
        o.add_sequence(s, True)
        out.append(o)
    return out


def assert_rows(coll, osk, what):
    rows = coll.rows_np()
    assert len(rows) == len(osk), what
    for s, (row, o) in enumerate(zip(rows, osk)):
        assert np.array_equal(row, o.mins_np()), (what, s, len(row), o.size())


def raw_call(buf, offsets, tpls):
    """The C call with an `out` array preset to non-NULL garbage; returns (error code or 0, out pointers)."""
    o = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = max(1, len(tpls))
    out = (C.c_void_p * n)(*([0x1234] * n))
    L = smb.lib()
    L.sourmash_err_clear()
    L.smgpu_sketch_collections(smb._vp(buf), smb._vp(o), o.size - 1, smb._handles(tpls), len(tpls), False, out)
    code = L.sourmash_err_get_last_code()
    L.sourmash_err_clear()
    return code, [out[i] for i in range(n)]


# ------------------------------------------------------------------------------------------------
# template sets, against the oracle and against the one-template calls
# ------------------------------------------------------------------------------------------------
F21, F31, F51 = (0, 21, False, 42, SCALED), (0, 31, False, 42, SCALED), (0, 51, False, 42, SCALED)
SETS = {
    "scaled_21_31_51": [F21, F31, F51],
    "num500_21_31_51": [(500, 21, False, 42, 0), (500, 31, False, 42, 0), (500, 51, False, 42, 0)],
    "pair_21_51": [F21, F51],
    "pair_31_51": [(500, 51, False, 42, 0), F31],
    "fused_generic_protein": [F51, F21, (0, 25, False, 42, SCALED), F31, (0, 30, True, 42, SCALED)],
    "protein_only": [(0, 31, True, 42, SCALED), (300, 24, True, 2**63 + 5, 0)],
    "two_seeds": [F21, (0, 31, False, 2**64 - 1, SCALED), F51],
    "duplicate": [F31, (200, 21, False, 7, 0), F31],
}


@pytest.mark.parametrize("name", list(SETS))
def test_template_sets_match_the_oracle(name):
    params = SETS[name]
    buf, offsets = ragged_batch(0x5EED3000 + len(name))
    seqs = seqs_of(buf, offsets)
    colls = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    assert len(colls) == len(params)
    for m, p in enumerate(params):
        osk = oracle_sketches(p, seqs)
        assert_rows(colls[m], osk, (name, m))
        num, k, prot, seed, mx = p
        if not prot:   # the one-template call gives the same rows
            one = smb.SketchCollection.sketch_sequences(buf, offsets, num, k, seed, mx)
            for x, y in zip(one.rows_np(), colls[m].rows_np()):
                assert np.array_equal(x, y), (name, m)
        else:          # ... and a protein collection compares as one built by pushing per-object sketches
            pushed = []
            for s in seqs:
                g = smb.KmerMinHash(num, k, True, seed, mx, False)
                g.add_sequence(s, True)
                pushed.append(g)
            ref = smb.SketchCollection.from_sketches(pushed)
            got, want = smb.compare_matrix(colls[m], colls[m]), smb.compare_matrix(ref, ref)
            for x, y in zip(got, want):
                assert np.array_equal(x, y), (name, m)
            oc, osz = orc.compare_matrix(osk, osk)
            assert np.array_equal(got[0], oc) and np.array_equal(got[1], osz)
    if name == "duplicate":
        for x, y in zip(colls[0].rows_np(), colls[2].rows_np()):
            assert np.array_equal(x, y)


def test_protein_against_dna_collection_is_a_mismatch():
    buf, offsets = ragged_batch(0x5EED3100)
    params = [(0, 30, True, 42, SCALED), (0, 30, False, 42, SCALED)]   # one ksize: the check after the ksize check
    prot, dna = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    for a, b in ((prot, dna), (dna, prot)):
        with pytest.raises(smb.SourmashError) as e:
            smb.compare_matrix(a, b)
        assert e.value.code == ERR_MISMATCH_DNAPROT


# ------------------------------------------------------------------------------------------------
# launches: one fused launch for 21/31/51 at one seed; one launch per template with fusion off
# ------------------------------------------------------------------------------------------------
def test_fused_launch_and_fusion_off():
    buf, offsets = ragged_batch(0x5EED3200)
    params = [F31, F51, F21]
    with counted() as c:
        fused = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    assert c["sketch_multi"] == 1 and sum(c.values()) == 1, c
    with counted() as c:
        mixed = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params + [(0, 25, False, 42, SCALED)]))
    assert c["sketch_multi"] == 1 and c["sketch_other"] == 1 and sum(c.values()) == 2, c
    smb.fuse_multi_k(False)
    try:
        with counted() as c:
            single = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    finally:
        smb.fuse_multi_k(True)
    assert c["sketch_k21"] == c["sketch_k31"] == c["sketch_k51"] == 1 and sum(c.values()) == 3, c
    seqs = seqs_of(buf, offsets)
    for m, p in enumerate(params):
        osk = oracle_sketches(p, seqs)
        for coll in (fused[m], mixed[m], single[m]):
            assert_rows(coll, osk, m)
    # unprofiled: the same rows
    again = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    for m in range(len(params)):
        for x, y in zip(again[m].rows_np(), fused[m].rows_np()):
            assert np.array_equal(x, y)


# ------------------------------------------------------------------------------------------------
# input variants
# ------------------------------------------------------------------------------------------------
def test_device_resident_input_and_empty_batch():
    import torch
    buf, offsets = ragged_batch(0x5EED3300)
    params = SETS["fused_generic_protein"] + [(300, 24, True, 9, 0)]
    host = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    t = torch.frombuffer(bytearray(buf + b"\0" * (-len(buf) % 16)), dtype=torch.uint8).cuda()
    to = torch.from_numpy(offsets.view(np.int64)).cuda()
    dev = smb.SketchCollection.sketch_sequences_multi(t.data_ptr(), to.data_ptr(), templates(params), on_device=True,
                                                      n_seqs=len(offsets) - 1)
    seqs = seqs_of(buf, offsets)
    for m, p in enumerate(params):
        assert_rows(dev[m], oracle_sketches(p, seqs), m)
        for x, y in zip(host[m].rows_np(), dev[m].rows_np()):
            assert np.array_equal(x, y), m
    for coll in smb.SketchCollection.sketch_sequences_multi(b"", [0], templates(params)):
        assert len(coll) == 0 and coll.rows_np() == []


# ------------------------------------------------------------------------------------------------
# survivor overflow of one template: only that one runs again
# ------------------------------------------------------------------------------------------------
def polya_input(n_polya, flank, seed):
    return random_dna(flank, seed) + b"A" * n_polya + random_dna(flank, seed + 1)


def polya_run(seq, k):
    """windows of seq whose canonical k-mer is poly-A (the one long A-run of seq; flanks are random)"""
    return max(len(m) for m in re.findall(rb"A+", seq)) - k + 1


@pytest.mark.parametrize("num, mx", [(0, MAX_HASH_1000), (50, 0)])
def test_survivor_overflow_of_one_template(num, mx):
    lens, parts = [], []
    for i in range(15):
        s = polya_input(40_000, 1000, 0x5EED3400 + i) if i % 5 == 2 else dirty(random_dna(3000, 0x5EED3500 + i), i)
        parts.append(s)
        lens.append(len(s))
    buf, offsets, n = b"".join(parts), offsets_of(lens), sum(lens)
    # the survivor reservation of sketch_many.cu and its threshold (the same for the three DNA templates)
    frac = mx / 2**64 if mx else min(1.0, 16.0 * num / float(np.median(lens)))
    thr = mx if mx else int(frac * 2**64)
    # a seed at which the poly-A 21-mer survives and the poly-A 31- and 51-mers do not
    seed = 99991
    while not (orc.hash_murmur(b"A" * 21, seed) <= min(thr, MAX_HASH_1000)
               and orc.hash_murmur(b"A" * 31, seed) > thr and orc.hash_murmur(b"A" * 51, seed) > thr):
        seed += 1
    assert sum(polya_run(s, 21) for s in parts if b"A" * 1000 in s) > frac * 1.25 * n + 4096
    params = [(num, k, False, seed, mx) for k in (21, 31, 51)]
    if num:   # every row keeps num hashes under the estimated threshold: no row is sketched again on its own
        for k in (21, 31, 51):
            for s in parts:
                o = orc.KmerMinHash(0, k, False, seed, thr, False)
                o.add_sequence(s, True)
                assert o.size() >= num
    with counted() as c:
        colls = smb.SketchCollection.sketch_sequences_multi(buf, offsets, templates(params))
    assert c["sketch_multi"] == 1 and c["sketch_k21"] == 1 and sum(c.values()) == 2, c
    for m, p in enumerate(params):
        assert_rows(colls[m], oracle_sketches(p, parts), m)


# ------------------------------------------------------------------------------------------------
# refusals: an error, every out[m] NULL
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case, code", [
    ("abundance", ERR_INTERNAL), ("neither_num_nor_max_hash", ERR_INTERNAL), ("num_and_max_hash", ERR_INTERNAL),
    ("dna_ksize_0", ERR_INTERNAL), ("protein_ksize_2", ERR_PANIC), ("no_templates", ERR_INTERNAL),
    ("seven_templates", ERR_INTERNAL)])
def test_refused_template_sets(case, code):
    buf, offsets = ragged_batch(0x5EED3600)
    good = [smb.KmerMinHash(0, 21, False, 42, SCALED, False), smb.KmerMinHash(0, 30, True, 42, SCALED, False)]
    bad = {
        "abundance": [smb.KmerMinHash(0, 31, False, 42, SCALED, True)],
        "neither_num_nor_max_hash": [smb.KmerMinHash(0, 31, False, 42, 0, False)],
        "num_and_max_hash": [smb.KmerMinHash(500, 31, False, 42, SCALED, False)],
        "dna_ksize_0": [smb.KmerMinHash(0, 0, False, 42, SCALED, False)],
        "protein_ksize_2": [smb.KmerMinHash(0, 2, True, 42, SCALED, False)],
        "no_templates": None,
        "seven_templates": [smb.KmerMinHash(0, k, False, 42, SCALED, False) for k in (21, 31, 51, 25, 33, 41, 61)],
    }[case]
    tpls = [] if bad is None else (bad if case == "seven_templates" else good + bad)
    got, out = raw_call(buf, offsets, tpls)
    assert got == code
    assert all(p is None for p in out[:len(tpls)]), out
    with pytest.raises(smb.SourmashError) as e:
        smb.SketchCollection.sketch_sequences_multi(buf, offsets, tpls)
    assert e.value.code == code
    # the templates are untouched and still usable
    coll, = smb.SketchCollection.sketch_sequences_multi(buf, offsets, good[:1])
    assert len(coll) == len(offsets) - 1
    assert all(t.size() == 0 for t in tpls)
