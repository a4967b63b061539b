"""Time one rank's row shard of the cfg3 all-vs-all matrix on one GPU for R = 1, 2, 4, 8 ranks, without and with
the probe form of the join (smgpu_compare_path 3, and 0 / 2: chosen from the data / forced)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import numpy as np, torch
import sourmash_rust_b200 as smb
from bench import planted_sketches
N, NUM = 10000, 500
rows = planted_sketches(N, NUM, 5)
offs = np.arange(N + 1, dtype=np.uint64) * np.uint64(NUM)
dev = torch.device("cuda", 0)
coll = smb.SketchCollection.from_csr(rows.reshape(-1), offs, N, NUM, 31)
for R in (1, 2, 4, 8):
    nr = N // R
    common = torch.empty((nr, N), dtype=torch.int32, device=dev); size = torch.empty_like(common)
    ratio = torch.empty((nr, N), dtype=torch.float64, device=dev)
    res = {}
    for path in ("noprobe", "auto", "sparse"):
        smb.compare_path(path)
        r0 = (R // 2) * nr if R > 1 else 0
        def step():
            smb.compare_matrix_device(coll, coll, "compare", r0, nr, 0, N, common.data_ptr(), size.data_ptr(), ratio.data_ptr(), N)
        step(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        st = torch.cuda.ExternalStream(smb._call("smgpu_stream"))
        e0.record(st)
        for _ in range(5):
            step()
        e1.record(st); torch.cuda.synchronize()
        res[path] = (e0.elapsed_time(e1) / 5, int(common.sum().item()))
        smb.profile_enable(True)
        for kind in ("join_sort", "compare"):
            smb.profile_read(kind, reset=True)
        step(); torch.cuda.synchronize()
        print("   R=%d %s: sort scope %.3f ms, join+walk scope %.3f ms" % (R, path, smb.profile_read("join_sort", True)[0],
                                                                          smb.profile_read("compare", True)[0]))
        smb.profile_enable(False)
    print("R=%d rows %d: noprobe %.3f ms, auto %.3f ms, sparse %.3f ms (checksums %d %d %d) -> whole matrix at R ranks: %.2e / %.2e pairs/s" % (
        R, nr, res["noprobe"][0], res["auto"][0], res["sparse"][0], res["noprobe"][1], res["auto"][1], res["sparse"][1],
        N * N / (res["noprobe"][0] * 1e-3), N * N / (res["auto"][0] * 1e-3)))
smb.compare_path("auto")
