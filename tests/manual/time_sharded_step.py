"""cfg3's sharded step (smgpu_compare_matrix_allgather: gather + this rank's row block) timed under torchrun:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
      tests/manual/time_sharded_step.py [reps=20]
Prints ms per step (max over ranks) and rank 0's kernel times; checks on every rank that the step gives the rows
[lo, hi) of the one-process matrix (smgpu_compare_matrix over the whole collection)."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import numpy as np, torch, torch.distributed as dist
import sourmash_rust_b200 as smb
from bench import planted_sketches

rank, world, local_rank = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
torch.cuda.set_device(local_rank)
smb.set_device(local_rank)
dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
smb.comm_init_from_torch()
dev = torch.device("cuda", local_rank)
N, NUM = 10000, 500
rows = planted_sketches(N, NUM, 0x5EED0100)
lo, hi = N * rank // world, N * (rank + 1) // world
nr = hi - lo
local = smb.SketchCollection.from_csr(rows[lo:hi].reshape(-1), np.arange(nr + 1, dtype=np.uint64) * np.uint64(NUM), nr, NUM, 31)
common = torch.empty((nr, N), dtype=torch.int32, device=dev)
size = torch.empty_like(common)
ratio = torch.empty((nr, N), dtype=torch.float64, device=dev)
# what the block must be: the same rows of the one-process matrix (no communicator involved)
whole = smb.SketchCollection.from_csr(rows.reshape(-1), np.arange(N + 1, dtype=np.uint64) * np.uint64(NUM), N, NUM, 31)
want = (torch.empty_like(common), torch.empty_like(size), torch.empty_like(ratio))
smb.compare_matrix_device(whole, whole, "compare", lo, nr, 0, N, want[0].data_ptr(), want[1].data_ptr(), want[2].data_ptr(), N)
torch.cuda.synchronize()
smb.profile_enable(True)
for i in range(3):
    smb.compare_matrix_allgather_device(local, "compare", common.data_ptr(), size.data_ptr(), ratio.data_ptr(), N)
for k in smb.PROFILE_KINDS:
    smb.profile_read(k, reset=True)
torch.cuda.synchronize()
dist.barrier()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for i in range(reps):
    smb.compare_matrix_allgather_device(local, "compare", common.data_ptr(), size.data_ptr(), ratio.data_ptr(), N)
e1.record()
torch.cuda.synchronize()
ms = torch.tensor([e0.elapsed_time(e1) / reps], device=dev)
dist.all_reduce(ms, op=dist.ReduceOp.MAX)
same = all(torch.equal(a, b) for a, b in zip(want, (common, size, ratio)))
kern = {k: round(smb.profile_read(k, reset=True)[0] / reps, 4) for k in ("join_sort", "compare", "compare_probe", "compare_fill", "compare_walk")}
if rank == 0:
    print("world %d: %.4f ms per step = %.3g pairs/s; rank 0 kernels %s; equals the one-process block: %s"
          % (world, ms.item(), N * N / (ms.item() * 1e-3), kern, same), flush=True)
assert same
# the exchange alone (header round trip + gather + wait), for the split of the step
for i in range(3):
    g = smb.collection_allgather(local)
torch.cuda.synchronize()
dist.barrier()
import time
t0 = time.perf_counter()
for i in range(reps):
    g = smb.collection_allgather(local)
    smb.device_sync() if hasattr(smb, "device_sync") else torch.cuda.synchronize()
t1 = time.perf_counter()
ms = torch.tensor([(t1 - t0) * 1e3 / reps], device=dev)
dist.all_reduce(ms, op=dist.ReduceOp.MAX)
if rank == 0:
    print("world %d: collection_allgather alone %.4f ms per call (host clock, synchronised)" % (world, ms.item()), flush=True)
smb.comm_destroy()
dist.destroy_process_group()
