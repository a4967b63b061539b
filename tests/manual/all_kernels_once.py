"""Small end-to-end run that launches every kernel family once (a quick check after kernel changes)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import sourmash_rust_b200 as smb
from util import MAX_HASH_1000, make_reads, random_dna, splitmix64
g = random_dna(30_000, 5)
reads = make_reads(g, 300, 150, 6)
mhs = [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000 * 20, True) for k in (21, 31, 51)]
smb.add_reads(mhs, reads, 300, 150, force=False)
smb.add_reads(mhs, reads, 300, 150, force=False)
print([m.size() for m in mhs], [m.md5sum()[:8] for m in mhs])
a, b = smb.KmerMinHash(200, 31, False, 42, 0, True), smb.KmerMinHash(200, 31, False, 42, 0, True)
a.add_sequence(g[:20000]); b.add_sequence(g[5000:25000])
print(a.compare(b), a.count_common(b))
c = smb.KmerMinHash(50, 9, False, 42, 0, False); c.add_sequence(g[:3000]); print(c.size())
p = smb.KmerMinHash(100, 30, True, 42, 0, False); p.add_sequence(g[:6000]); print(p.size())
sk = []
for i in range(40):
    m = smb.KmerMinHash(100, 21, False, 42, 0, False); m.add_sequence(g[i * 300:i * 300 + 6000]); sk.append(m)
coll = smb.SketchCollection.from_sketches(sk)
for path in ("auto", "dense"):
    smb.compare_path(path)
    cm, sz, r = smb.compare_matrix(coll, coll, "compare")
    cm2, _, _ = smb.compare_matrix(coll, coll, "containment", r0=3, nr=9)
    print(path, int(cm.sum()), int(cm2.sum()))
smb.compare_path("auto")
print(len(smb.linear_find(coll, smb.SketchCollection.from_sketches(sk[:5]), "containment", 0.1)))
ng = smb.Nodegraph([997, 1009], 21)
print(ng.count_many(splitmix64(1, 500))[0], ng.get_many(splitmix64(1, 600))[0])
