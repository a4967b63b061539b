"""The canonical-strand choice at the inputs random reads almost never reach, bit for bit against the oracle.

The sketch kernels pick the strand of a k-mer by comparing the 2-bit words of the forward and reverse-complement
k-mers, most significant word first (kmer_bits.cuh, canonical_is_fw): the top word holds the last 16 bases of
each strand, and the last bases of the reverse complement are the complemented first bases of the forward k-mer.
So a k-mer whose last m bases are the reverse complement of its first m bases (a near-palindrome) ties on the
top 2m bits, and the comparison is decided at base m.  Random k-mers decide in the top word 15 times in 16; at
k = 51 (four words, one borrow chain on the device) a near-palindrome with m >= 16 ties the whole top word.  For
odd k the middle base is never its own complement, so every m up to (k - 1) / 2 is reachable and none ties fully.

Every m from 0 to (k - 1) / 2 is built, with each of the three mismatching bases at position m (so both strands
win), inside random flanks, for k = 21, 31 and 51 alone and in every fused group, at two seeds, into sketches
that keep every hash."""
import numpy as np
import pytest

import sourmash_rust_b200 as smb
from test_gpu_sketch_edges import counted, offsets_of, oracle_batch, pair, same
from util import splitmix64

pytestmark = pytest.mark.gpu

KEEP_ALL = 2**64 - 1          # scaled sketch whose threshold passes every hash
COMP = {"A": "T", "C": "G", "G": "C", "T": "A"}
GROUPS = [(21,), (31,), (51,), (21, 31), (21, 51), (31, 51), (21, 31, 51)]


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


def near_palindrome(k, m, mismatch, rnd):
    """a k-mer whose last m bases are the reverse complement of its first m, and whose base k - 1 - m is the
    `mismatch`-th (0..2) base other than the complement of base m"""
    bases = ["ACGT"[int(x) & 3] for x in rnd[:k]]
    for i in range(m):
        bases[k - 1 - i] = COMP[bases[i]]
    others = [b for b in "ACGT" if b != COMP[bases[m]]]
    bases[k - 1 - m] = others[mismatch]
    return "".join(bases)


def top_words_tied(kmer):
    """top 32-bit words equal in the end-aligned 2-bit encodings of the two strands (kmer_bits.cuh extract2_end)"""
    k = len(kmer)
    ne = (2 * k + 31) // 32
    pad = 16 * ne - k
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    rc = "".join(COMP[b] for b in reversed(kmer))
    ef = sum(code[b] << (2 * (j + pad)) for j, b in enumerate(kmer))
    er = sum(code[b] << (2 * (j + pad)) for j, b in enumerate(rc))
    tied = 0
    for w in reversed(range(ne)):
        if (ef >> (32 * w)) & 0xFFFFFFFF != (er >> (32 * w)) & 0xFFFFFFFF:
            break
        tied += 1
    return tied


def near_palindrome_batch(ks, seed):
    """one sequence per (k, m, mismatch, copy): random flank of 0..24 bases, the near-palindrome, random flank"""
    seqs, tied = [], {}
    r = splitmix64(seed, 1 << 20)
    pos = 0
    for k in ks:
        for m in range((k - 1) // 2 + 1):
            for mismatch in range(3):
                for _ in range(2):
                    left, right = int(r[pos]) % 25, int(r[pos + 1]) % 25
                    pos += 2
                    flank = "".join("ACGT"[int(x) & 3] for x in r[pos:pos + left + right])
                    pos += left + right
                    kmer = near_palindrome(k, m, mismatch, r[pos:pos + k])
                    pos += k
                    seqs.append(flank[:left] + kmer + flank[left:])
                    tied[k] = max(tied.get(k, 0), top_words_tied(kmer))
    lens = [len(s) for s in seqs]
    return "".join(seqs).encode(), offsets_of(lens), tied


@pytest.mark.parametrize("seed", [42, 2**64 - 1])
@pytest.mark.parametrize("ks", GROUPS, ids=lambda ks: "k" + "_".join(map(str, ks)))
def test_near_palindromes_pick_the_oracle_strand(ks, seed):
    buf, offsets, tied = near_palindrome_batch((21, 31, 51), 0x7A1E0000 + seed % 1000)
    # the batch reaches the deepest tie each k allows: the whole top word at k = 51, none at 21 and 31
    assert tied == {21: 0, 31: 0, 51: 1}
    gos = [pair(0, k, KEEP_ALL, True, seed) for k in ks]
    with counted() as n:
        smb.add_sequences([g for g, _ in gos], buf, offsets)
    kind = "sketch_multi" if len(ks) > 1 else "sketch_k%d" % ks[0]
    assert n[kind] == 1 and sum(n.values()) == 1, n
    oracle_batch([o for _, o in gos], buf, offsets, True)
    for g, o in gos:
        assert g.size() > 0
        same(g, o)
    # and every constructed k-mer is in the sketch: the batch keeps each window's hash
    n_windows = sum(max(0, int(offsets[s + 1] - offsets[s]) - k + 1) for k in ks for s in range(len(offsets) - 1))
    assert sum(int(g.abunds_np().sum()) for g, _ in gos) == n_windows
