"""Host batches of many chunks, against the oracle (tests/test_gpu_sketch_edges.py starts this with
SMB200_H2D_CHUNK_MB=1: the library reads the chunk size once, when it loads).

add_sequences copies a host batch to the device in chunks and launches the sketch kernels for the tiles each chunk
completes.  Here the chunk size is small enough for a 6 MiB batch to cross six chunk edges, with sequence ends on
every side of each edge, a k-mer across an edge, and the first invalid base in the last chunk.  Launch counts follow
from CHUNK below, so this fails (rather than passing without reaching the edges) if the library runs another chunk
size.  Prints "ok" at the end."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import sourmash_rust_b200 as smb  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from test_gpu_sketch_edges import (chunk_ends, counted, dirty, gpu_batch, offsets_of, oracle_batch, pair,  # noqa: E402
                                   polya_input, polya_run, polya_seed, same, six_sketches, sketch_launches)
from util import MAX_HASH_1000, make_reads, random_dna, splitmix64  # noqa: E402

CHUNK = 1 << 20
N_EDGES = 6
STRADDLE = 3   # the chunk edge that one long sequence crosses (no short sequences there)
EDGE_ENDS = [-52, -51, -50, -33, -32, -31, -30, -22, -21, -20, -2, -1, 0, 1, 2, 20, 21, 22, 30, 31, 32, 33, 50, 51, 52]


def ragged_batch():
    """About 6 MiB of sequence lengths: at every chunk edge but STRADDLE, sequences end at each offset of EDGE_ENDS
    (-k-1 .. +k+1 for k = 21, 31, 33, 51 and the protein k 30); at STRADDLE one sequence crosses the edge and ends 40
    bytes after it.  Between edges, a few long sequences of random length."""
    n = N_EDGES * CHUNK + 12345
    r = splitmix64(0x5EED2000, 4 * N_EDGES)
    ends = []
    for j in range(1, N_EDGES + 1):
        e = j * CHUNK
        ends += [(j - 1) * CHUNK + 100 + int(x % np.uint64(CHUNK - 300)) for x in r[3 * j:3 * j + 3]]
        ends += [e + 40] if j == STRADDLE else [e + d for d in EDGE_ENDS]
    ends = sorted(set(ends)) + [n]
    return np.diff([0] + ends)


def launches_of(ends, fused_k, singles):
    """expected counts: one fused launch per chunk for the group (its widest k), one per chunk for each single k"""
    want = {"sketch_k21": 0, "sketch_k31": 0, "sketch_k51": 0, "sketch_other": 0, "sketch_multi": 0}
    if fused_k:
        want["sketch_multi"] = sketch_launches(fused_k, ends)
    for k in singles:
        want[{21: "sketch_k21", 31: "sketch_k31", 51: "sketch_k51"}.get(k, "sketch_other")] += sketch_launches(k, ends)
    return want


def run_twice(make, call, os_, want):
    """make() -> fresh device sketches; call(gs) runs the batch.  Once profiled (launch counts == want), once with
    each sketch on its own stream; both equal the oracle sketches os_."""
    for profiled in (True, False):
        gs = make()
        if profiled:
            with counted() as c:
                r = call(gs)
            assert c == want, (c, want)
        else:
            r = call(gs)
        for g, o in zip(gs, os_):
            same(g, o)
        yield r


lens = ragged_batch()
offsets = offsets_of(lens)
n = int(offsets[-1])
ends = chunk_ends(n, CHUNK)
assert len(ends) == N_EDGES + 1 and ends[:-1] == [j * CHUNK for j in range(1, N_EDGES + 1)]
clean = random_dna(n, 0x5EED2001)

# ---- six sketches, force = true, dirty input -------------------------------------------------------------------
buf = dirty(clean, 0x5EED2002, n_bad=400)
os_ = [o for _, o in six_sketches(2**63)]
oracle_batch(os_, buf, offsets, True)
list(run_twice(lambda: [g for g, _ in six_sketches(2**63)], lambda gs: smb.add_sequences(gs, buf, offsets, force=True),
               os_, launches_of(ends, 51, [31, 33])))
print("six sketches, force=true: ok")

# ---- force = false: one invalid base (a) in the last chunk, (b) in k-mers across the edge STRADDLE -------------------
for where in (n - 1000, STRADDLE * CHUNK - 3):
    s = int(np.searchsorted(offsets, where, side="right")) - 1
    if where > ends[-2]:   # (a)
        assert offsets[s] < where - 51
    else:                  # (b): the sequence holding it starts 51 bases before it and crosses the edge
        assert offsets[s] < where - 51 and offsets[s + 1] == STRADDLE * CHUNK + 40
    a = bytearray(clean)
    a[where] = ord("N")
    bad = bytes(a)
    os_ = [o for _, o in six_sketches(2**63)]
    msg = oracle_batch(os_, bad, offsets, False)
    assert msg.split(": ")[1] == bad[where - 20:where + 1].decode()   # the first sketch (k = 21) reports
    # every DNA sketch runs once more up to its first failing k-mer
    want = launches_of(ends, 51, [31, 33])
    for kd, extra in (("sketch_k21", 1), ("sketch_k31", 2), ("sketch_k51", 1), ("sketch_other", 1)):
        want[kd] += extra
    for got in run_twice(lambda: [g for g, _ in six_sketches(2**63)], lambda gs: gpu_batch(gs, bad, offsets, False),
                         os_, want):
        assert got == msg, (got, msg)
print("force=false: ok")

# ---- one fused pair at seed 42 and k = 51 at seed 7 ---------------------------------------------------------------
spec = ((21, 42), (31, 42), (51, 7))
os_ = [pair(0, k, MAX_HASH_1000 * 20, True, s)[1] for k, s in spec]
oracle_batch(os_, buf, offsets, True)
list(run_twice(lambda: [pair(0, k, MAX_HASH_1000 * 20, True, s)[0] for k, s in spec],
               lambda gs: smb.add_sequences(gs, buf, offsets, force=True), os_, launches_of(ends, 31, [51])))
print("mixed seeds: ok")

# ---- fixed-length reads, ASCII and 2-bit ----------------------------------------------------------------------------
read_len = 151
n_reads = N_EDGES * CHUNK // read_len + 7
reads = make_reads(random_dna(1_000_000, 0x5EED2003), n_reads, read_len, 0x5EED2004)
ks = [21, 31, 51]
os_ = orc.mt_sketch_reads(reads, n_reads, read_len, ks, 0, MAX_HASH_1000, True, os.cpu_count() or 4)
mk = lambda: [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000, True) for k in ks]  # noqa: E731
r_ends = chunk_ends(n_reads * read_len, CHUNK)
assert len(r_ends) > N_EDGES
list(run_twice(mk, lambda gs: smb.add_reads(gs, reads, n_reads, read_len, force=False), os_, launches_of(r_ends, 51, [])))
packed = smb.pack_2bit(np.frombuffer(reads, dtype=np.uint8), read_len)
p_ends = chunk_ends(n_reads * read_len, CHUNK, packed_read_len=read_len)
assert len(p_ends) > N_EDGES and all(e % read_len == 0 for e in p_ends)
list(run_twice(mk, lambda gs: smb.add_reads_2bit(gs, packed, n_reads, read_len), os_, launches_of(p_ends, 51, [])))
print("reads: ok")

# ---- re-runs after a batch of several chunks: overflow (scaled), overflow + estimate widening (num) -------------------
k = 21
seed = polya_seed(k, 2**40)
seq = polya_input(5 * CHUNK // 2, 5000, 0x5EED2005)
n_p = len(seq)
p_ends = chunk_ends(n_p, CHUNK)
assert len(p_ends) >= 3
windows = polya_run(seq, k)
assert windows > MAX_HASH_1000 / 2**64 * 1.25 * n_p + 4096
o = orc.KmerMinHash(0, k, False, seed, MAX_HASH_1000, True)
o.add_sequence(seq, True)
want = launches_of(p_ends, 0, [k])
want["sketch_k21"] += 1
list(run_twice(lambda: [smb.KmerMinHash(0, k, False, seed, MAX_HASH_1000, True)],
               lambda gs: smb.add_sequences(gs, seq, [0, n_p]), [o], want))
num = 5000
est = 8.0 * num + 4096.0
assert n_p > 4 * est and est / n_p > 2.0**-6   # the estimate is used, and one widening reaches the whole hash range
o_est = orc.KmerMinHash(0, k, False, seed, int(est / n_p * 2**64), False)
o_est.add_sequence(seq, True)
assert o_est.size() < num and windows > est * 1.25 + 4096
o = orc.KmerMinHash(num, k, False, seed, 0, True)
o.add_sequence(seq, True)
want["sketch_k21"] += 1
list(run_twice(lambda: [smb.KmerMinHash(num, k, False, seed, 0, True)],
               lambda gs: smb.add_sequences(gs, seq, [0, n_p]), [o], want))
print("re-runs: ok")
print("ok")
