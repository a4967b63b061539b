"""One smgpu_sketch_collections call against one smgpu_sketch_collection call per template.

N synthetic genomes (default 128 x 5 Mbp = 640 MB, more than the 126 MB of L2; SplitMix64 bases as in tests/util.py)
are sketched with k = 21/31/51 at scaled = 1000, from page-locked host memory and from device memory:
  one   = one call with the three templates (one host-to-device copy, the fused k = 21/31/51 kernel)
  three = three calls, one per k-size (three copies of a host batch, three single-k kernels)
and in a third leg with a translated protein template (k = 30, scaled = 1000) added, where the separate form builds the
protein collection the only other way there is: one add_sequence per genome, then a push.
Each time is a host clock around one form, ending in a device synchronise, after a warm-up of every form; the forms
alternate within each of --reps repetitions.  The rows of both forms must be equal.

usage: bench_sketch_collections.py --out DIR [--genomes 128] [--length 5000000] [--reps 5]
Writes DIR/bench_sketch_collections.json with the GPU's name and power limit read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch

import sourmash_rust_b200 as smb
from util import MAX_HASH_1000, random_dna

ap = argparse.ArgumentParser()
ap.add_argument("--out", required=True)
ap.add_argument("--genomes", type=int, default=128)
ap.add_argument("--length", type=int, default=5_000_000)
ap.add_argument("--reps", type=int, default=5)
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("no CUDA device: this script measures on the GPU only")
N, L = args.genomes, args.length
assert L % 16 == 0

from sourmash_rust_b200 import build
build.build_library()
dev = torch.device("cuda", 0)
name = torch.cuda.get_device_name(0)
power = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip()

host = torch.empty(N * L, dtype=torch.uint8, pin_memory=True)
for i in range(N):
    host[i * L:(i + 1) * L] = torch.from_numpy(np.frombuffer(random_dna(L, 0x5EED4000 + i), dtype=np.uint8))
offsets = (np.arange(N + 1, dtype=np.uint64) * np.uint64(L))
dbuf = host.to(dev)
doff = torch.from_numpy(offsets.view(np.int64)).to(dev)
one_off_d = torch.tensor([0, L], dtype=torch.int64, device=dev)
one_off_h = np.array([0, L], dtype=np.uint64)
torch.cuda.synchronize()

DNA = [(0, k, False, 42, MAX_HASH_1000) for k in (21, 31, 51)]
PROT = (0, 30, True, 42, MAX_HASH_1000)


def inputs(on_device):
    return (dbuf.data_ptr(), doff.data_ptr()) if on_device else (host.data_ptr(), offsets)


def one_call(params, on_device):
    b, o = inputs(on_device)
    tpls = [smb.KmerMinHash(*p) for p in params]
    return smb.SketchCollection.sketch_sequences_multi(b, o, tpls, on_device=on_device, n_seqs=N)


def separate(params, on_device):
    b, o = inputs(on_device)
    out = []
    for num, k, prot, seed, mx in params:
        if not prot:
            out.append(smb.SketchCollection.sketch_sequences(b, o, num, k, seed, mx, on_device=on_device, n_seqs=N))
            continue
        coll = smb.SketchCollection()
        for i in range(N):
            m = smb.KmerMinHash(num, k, True, seed, mx, False)
            if on_device:
                m.add_sequences(dbuf.data_ptr() + i * L, one_off_d.data_ptr(), on_device=True, n_seqs=1)
            else:
                m.add_sequences(host.data_ptr() + i * L, one_off_h)
            coll.push(m)
        out.append(coll)
    return out


def timed(fn, *a):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn(*a)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def rows(colls):
    return [c.rows_np() for c in colls]


legs = []
for leg, params, on_device in (("host_dna", DNA, False), ("device_dna", DNA, True), ("host_dna_protein", DNA + [PROT], False),
                               ("device_dna_protein", DNA + [PROT], True)):
    _, a = timed(one_call, params, on_device)    # warm-up of both forms, and the check that they agree
    _, b = timed(separate, params, on_device)
    for m, (x, y) in enumerate(zip(rows(a), rows(b))):
        assert len(x) == len(y) == N
        for s in range(N):
            assert np.array_equal(x[s], y[s]), (leg, m, s)
    hashes = sum(sum(len(r) for r in rr) for rr in rows(a))
    del a, b
    t_one, t_sep = [], []
    for rep in range(args.reps):
        t, r = timed(one_call, params, on_device)
        t_one.append(t)
        del r
        t, r = timed(separate, params, on_device)
        t_sep.append(t)
        del r
    res = {"leg": leg, "templates": ["%s k=%d" % ("protein" if p[2] else "dna", p[1]) for p in params], "on_device": on_device,
           "one_call_ms": [round(t * 1e3, 3) for t in t_one], "separate_ms": [round(t * 1e3, 3) for t in t_sep],
           "one_call_median_ms": round(statistics.median(t_one) * 1e3, 3),
           "separate_median_ms": round(statistics.median(t_sep) * 1e3, 3),
           "speedup_median": round(statistics.median(t_sep) / statistics.median(t_one), 3), "hashes": hashes}
    print(json.dumps(res), flush=True)
    legs.append(res)

out = {"gpu": name, "power_limit": power, "genomes": N, "length": L, "bytes": N * L, "reps": args.reps, "legs": legs}
os.makedirs(args.out, exist_ok=True)
with open(os.path.join(args.out, "bench_sketch_collections.json"), "w") as f:
    json.dump(out, f, indent=1)
print(json.dumps({k: v for k, v in out.items() if k != "legs"}))
