"""The sketch kernels' threshold test at the hash values it has to separate, bit for bit against the oracle.

The k-mer loops test the high words of the two MurmurHash3 addends first and finish the hash only for the windows
that may pass (sketch.cu, kmer_loop).  So a scaled sketch is built here with max_hash set to hashes that occur in the
input, one below them, a value sharing a hash's high word with a lower low word, and near 2^64 (a threshold whose
high word is 2^32 - 1, where every window passes the first test), for k = 21, 31 and 51 alone and fused, at two
seeds."""
import numpy as np
import pytest

import sourmash_rust_b200 as smb
from oracle import oracle as orc
from test_gpu_sketch_edges import offsets_of, oracle_batch, pair, same
from util import random_dna

pytestmark = pytest.mark.gpu

GROUPS = [(21,), (31,), (51,), (21, 31, 51)]


@pytest.fixture(scope="module", autouse=True)
def _built():
    from sourmash_rust_b200 import build
    build.build_library()
    smb.lib()


def thresholds(buf, offsets, k, seed):
    """max_hash values at and around the hashes of the input"""
    o = orc.KmerMinHash(0, k, False, seed, 2**64 - 1, False)
    oracle_batch([o], buf, offsets, True)
    h = [int(x) for x in o.mins_np()]
    picks = [h[0], h[1], h[len(h) // 1000], h[len(h) // 100], h[len(h) // 10], h[len(h) // 2], h[-1]]
    out = set()
    for x in picks:
        out.update({x, x - 1, (x >> 32) << 32})
    out.update({2**64 - 2, 2**64 - 2**32, 2**64 - 2**32 - 1})
    return sorted(v for v in out if v > 0)


@pytest.mark.parametrize("seed", [42, 7])
@pytest.mark.parametrize("ks", GROUPS, ids=lambda ks: "k" + "_".join(map(str, ks)))
def test_scaled_thresholds_at_hash_values(ks, seed):
    lens = [5000, 21, 51, 3000, 151, 151, 800]
    offsets = offsets_of(lens)
    buf = random_dna(int(offsets[-1]), 0x7E5E0000 + seed)
    per_k = {k: thresholds(buf, offsets, k, seed) for k in ks}
    for i in range(max(len(v) for v in per_k.values())):
        gos = [pair(0, k, per_k[k][min(i, len(per_k[k]) - 1)], True, seed) for k in ks]
        smb.add_sequences([g for g, _ in gos], buf, offsets)
        oracle_batch([o for _, o in gos], buf, offsets, True)
        for g, o in gos:
            same(g, o)
    # the picks include a threshold equal to a hash, so the inclusive bound was exercised
    for k in ks:
        assert any(t + 1 in per_k[k] for t in per_k[k])
    assert np.uint64(per_k[ks[0]][-1]) >> np.uint64(32) == np.uint64(0xFFFFFFFF)
