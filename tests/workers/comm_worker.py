"""One rank of the multi-GPU parity check (tests/test_gpu_comm.py starts WORLD of these, one per GPU; also runs
stand-alone with WORLD=1).  Every rank derives ALL ranks' inputs from the same seeds, takes its share, runs the
library's collective entry points (include/sourmash_b200.h, comm.cu: NCCL inside the library) and compares with
what one process computes over the whole input -- and with the CPU oracle.

env: RANK, WORLD, LOCAL_RANK, COMM_ID_FILE (rank 0 writes the 128-byte NCCL id there, the others wait for it)."""
import os
import sys
import time

import numpy as np
import torch  # before the library binds NCCL: the process then has ONE libnccl.so.2 (torch's), found by SONAME

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import sourmash_rust_b200 as smb  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from util import MAX_HASH_1000, make_reads, random_dna, splitmix64  # noqa: E402

rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD", 1))
smb.set_device(int(os.environ.get("LOCAL_RANK", rank)))
id_file = os.environ["COMM_ID_FILE"]
if rank == 0:
    with open(id_file + ".tmp", "wb") as f:
        f.write(smb.comm_unique_id())
    os.rename(id_file + ".tmp", id_file)
else:
    t0 = time.time()
    while not os.path.exists(id_file):
        assert time.time() - t0 < 120, "no id file"
        time.sleep(0.05)
if os.environ.get("NO_COMM") == "1":   # a world of one needs no communicator: the collectives must act the same
    assert world == 1
else:
    smb.comm_init(open(id_file, "rb").read(), rank, world)
assert smb.comm_rank_world() == (rank, world)


def rows_for(kind, n_rows, seed):
    """n_rows sorted distinct rows; clusters of 8 share most hashes (so that pairs are related)."""
    out = []
    for i in range(n_rows):
        root = splitmix64(seed + i // 8, 700)
        own = splitmix64(seed * 7919 + i, 300)
        if kind == "num":
            r = np.unique(np.concatenate([root[: 500 + (i % 5) * 20], own[:60]]) >> np.uint64(3))[:200]
        else:
            r = np.unique(np.concatenate([root[: 300 + (i % 7) * 40], own[: 20 + (i * 13) % 200]]) % np.uint64(MAX_HASH_1000))
        out.append(r.astype(np.uint64))
    return out


def collection(rows, num, mx):
    offs = np.zeros(len(rows) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(r) for r in rows])
    h = np.concatenate(rows) if rows else np.zeros(0, dtype=np.uint64)
    return smb.SketchCollection.from_csr(h, offs, len(rows), num, 31, 42, mx)


def share(n, r):
    """uneven on purpose: rank r owns rows [lo, hi); one rank may own nothing"""
    cuts = [0] + [min(n, (n * (k + 1)) // world + (3 if k % 2 == 0 else -3) * (k < world - 1)) for k in range(world)]
    cuts[-1] = n
    return cuts[r], cuts[r + 1]


for kind, num, mx, n_rows in (("num", 200, 0, 96), ("scaled", 0, MAX_HASH_1000, 61), ("num", 200, 0, world - 1 if world > 1 else 1)):
    rows = rows_for(kind, n_rows, 1234 + n_rows)
    lo, hi = (share(n_rows, rank) if n_rows >= 4 * world else (min(rank, n_rows), min(rank + 1, n_rows)))
    local = collection(rows[lo:hi], num, mx)
    whole = collection(rows, num, mx)
    # 1. all-gather of the packed rows
    g = smb.collection_allgather(local)
    got = g.rows_np()
    assert len(got) == n_rows and all(np.array_equal(a, b) for a, b in zip(got, rows)), (kind, "allgather")
    # 2. this rank's row block, gather overlapped with the local table build, against the one-process matrix
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
    for mode in ("compare", "containment"):
        # (the sparse path over uniform rows starts the block while the gathered columns are still arriving)
        for path in ("auto", "sparse", "dense"):
            smb.compare_path(path)
            nr = hi - lo
            common = torch.full((max(1, nr), n_rows), -1, dtype=torch.int32, device=dev)
            size = torch.full((max(1, nr), n_rows), -1, dtype=torch.int32, device=dev)
            ratio = torch.full((max(1, nr), n_rows), -1.0, dtype=torch.float64, device=dev)
            g2 = smb.compare_matrix_allgather_device(local, mode, common.data_ptr(), size.data_ptr(), ratio.data_ptr(), n_rows)
            assert len(g2) == n_rows
            if nr:
                wc, ws, wr = smb.compare_matrix(whole, whole, mode, r0=lo, nr=nr)
                assert np.array_equal(common.cpu().numpy()[:nr].astype(np.uint32), wc), (kind, mode, path)
                assert np.array_equal(size.cpu().numpy()[:nr].astype(np.uint32), ws), (kind, mode, path)
                assert np.array_equal(ratio.cpu().numpy()[:nr], wr, equal_nan=True), (kind, mode, path)
        smb.compare_path("auto")
    # ... and against the oracle (first rows of the block)
    if hi > lo:
        osk = []
        for r in rows:
            o = orc.KmerMinHash(num, 31, False, 42, mx)
            o.add_many(r)
            osk.append(o)
        oc, osz = orc.compare_matrix(osk[lo:lo + 4], osk)
        wc, ws, _ = smb.compare_matrix(g, g, "compare", r0=lo, nr=min(4, hi - lo))
        assert np.array_equal(wc, oc[: wc.shape[0]].astype(np.uint32)) and np.array_equal(ws, osz[: ws.shape[0]].astype(np.uint32))
    # 4. partitioned linear index
    if n_rows >= 8:
        queries = collection([rows[3], rows[n_rows // 2], np.zeros(0, dtype=np.uint64), rows[n_rows - 1][::2].copy()], num, mx)
        for mode in ("similarity", "containment"):
            for thr in (0.0, 0.1, 0.5):
                want = smb.linear_find(whole, queries, mode, thr)
                got = smb.linear_find_sharded(local, queries, mode, thr, hits_cap=4 * n_rows)
                assert got == want, (kind, mode, thr, got, want)

# 3. partial sketches of one sample -> merged on every rank (cfg2's combine step)
genome = random_dna(300_000, 99)
for num, mx, ab in ((0, MAX_HASH_1000 * 20, True), (0, MAX_HASH_1000 * 20, False), (300, 0, True), (300, 0, False)):
    parts = []
    for r in range(world):
        o = orc.KmerMinHash(num, 21, False, 42, mx, ab)
        rd = make_reads(genome, 2000 + 100 * r, 150, 500 + r)
        o.add_reads(rd, len(rd) // 150, 150)
        parts.append((o, rd))
    mine = smb.KmerMinHash(num, 21, False, 42, mx, ab)
    mine.add_reads(parts[rank][1], len(parts[rank][1]) // 150, 150)
    smb.comm_allmerge(mine)
    acc = parts[0][0]
    for r in range(1, world):
        acc.merge(parts[r][0])
    assert np.array_equal(mine.mins_np(), acc.mins_np()), ("allmerge mins", num, mx, ab)
    if world > 1 or ab:
        ga, oa = mine.abunds_np(), acc.abunds_np()
        assert (ga is None) == (oa is None) and (ga is None or np.array_equal(ga, oa)), ("allmerge abunds", num, mx, ab)

smb.comm_destroy()
print("rank %d/%d ok (NCCL %d)" % (rank, world, smb.lib().smgpu_comm_nccl_version()), flush=True)
