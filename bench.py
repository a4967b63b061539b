#!/usr/bin/env python
"""bench.py -- sketch-and-compare hot path on N B200s (one process per GPU), or the reference
algorithm's CPU path on the host cores (--impl reference).

Workload (BASELINE.json configs[1], "cfg2"): scaled=1000 (max_hash = 18446744073709552), multi-k
k=21/31/51, synthetic error-free 150 bp reads from a random-ACGT genome, track_abundance.  One
step = one batch of READS_PER_STEP reads added to the three sketches (a batch is 315 MB of ASCII,
larger than the 126 MB L2).  Metric: Gbp/s sketched = input bases per second (every base is
sketched at all three k).  A second section times the all-vs-all Jaccard matrix of configs[2]
("cfg3": 10,000 sketches, num=500, k=31) and reports comparisons/s.

Prints ONE JSON line on rank 0 (see the keys below).  Timing: CUDA events on the library's own
stream (wrapped as a torch ExternalStream), barrier + synchronize on both sides, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MAX_HASH_1000 = 18446744073709552
KSIZES = (21, 31, 51)
READ_LEN = 150
GENOME_LEN = 100_000_000
SEED_GENOME = 0x5EED0010
SEED_READS = 0x5EED0011
# Executed SASS thread-instructions per window, DRAM bytes per window and pipe utilisations of the sketch kernels come
# from the ncu --set full captures, through profiles/kernel_constants.json (written by tests/manual/ncu_summary.py
# --json from the same report the committed summary table is made of) -- not pasted here, so they cannot go stale
# silently: a kernel the file does not list gets nulls.
KERNEL_OF = {21: "sketch_kernel<21,0,0>", 31: "sketch_kernel<31,0,0>", 51: "sketch_kernel<51,0,0>", "multi": "sketch_kernel<21,31,51>"}


def kernel_constants():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "kernel_constants.json")))
    except (OSError, ValueError):
        return {}


# ----------------------------------------------------------------------------------------------
# --dump-outputs: what the timed paths return to their caller, for comparing two builds output for output
# ----------------------------------------------------------------------------------------------
DUMP_MAX_BYTES = 64 << 20
DUMP_COMPARE_CELLS = 1 << 20   # at most this many of the parity check's seeded sample of matrix cells


def hash_words(h):
    """uint64 hashes as an (n, 2) float64 array of their high and low 32-bit halves: exact, where one float64 per
    hash would round every hash above 2**53"""
    return np.stack([(h >> np.uint64(32)).astype(np.float64), (h & np.uint64(0xFFFFFFFF)).astype(np.float64)], axis=1)


def dump_outputs(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, "outputs to dump are %d bytes, more than %d" % (total, DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ----------------------------------------------------------------------------------------------
# synthetic inputs
# ----------------------------------------------------------------------------------------------
def np_genome(n, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n, dtype=np.uint8)]


def np_reads(genome, n_reads, seed):
    """error-free reads, uniform start, strand flipped w.p. 0.5 (SURVEY 8(d) cfg2)"""
    rng = np.random.Generator(np.random.PCG64(seed))
    out = np.empty((n_reads, READ_LEN), dtype=np.uint8)
    comp = np.zeros(256, dtype=np.uint8)
    comp[list(b"ACGT")] = list(b"TGCA")
    ar = np.arange(READ_LEN, dtype=np.int64)
    for lo in range(0, n_reads, 1 << 18):
        hi = min(n_reads, lo + (1 << 18))
        starts = rng.integers(0, len(genome) - READ_LEN, size=hi - lo, dtype=np.int64)
        flips = rng.integers(0, 2, size=hi - lo, dtype=np.uint8).astype(bool)
        r = genome[starts[:, None] + ar[None, :]]
        r[flips] = comp[r[flips][:, ::-1]]
        out[lo:hi] = r
    return out.reshape(-1)


def torch_reads(genome_t, n_reads, seed, device):
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    out = torch.empty((n_reads, READ_LEN), dtype=torch.uint8, device=device)
    comp = torch.zeros(256, dtype=torch.uint8, device=device)
    comp[torch.tensor(list(b"ACGT"), device=device, dtype=torch.long)] = torch.tensor(list(b"TGCA"), dtype=torch.uint8, device=device)
    ar = torch.arange(READ_LEN, device=device)
    for lo in range(0, n_reads, 1 << 19):
        hi = min(n_reads, lo + (1 << 19))
        starts = torch.randint(0, genome_t.numel() - READ_LEN, (hi - lo,), generator=g, device=device)
        flips = torch.randint(0, 2, (hi - lo,), generator=g, device=device).bool()
        r = genome_t[starts[:, None] + ar[None, :]]
        rc = comp[r.flip(1).long()]
        out[lo:hi] = torch.where(flips[:, None], rc, r)
    return out.reshape(-1)


def planted_sketches(n_rows, num, seed):
    """cfg3 compare-only input (SURVEY 8(d)): 100-member clusters; a member keeps each hash of its
    cluster root with the k-mer survival probability of its substitution rate and fills up with
    fresh hashes; rows are the `num` smallest, sorted, distinct."""
    rng = np.random.Generator(np.random.PCG64(seed))
    rates = (0.001, 0.005, 0.01, 0.02, 0.05)
    rows = np.empty((n_rows, num), dtype=np.uint64)
    i = 0
    while i < n_rows:
        root = np.unique(rng.integers(0, 1 << 52, size=4 * num, dtype=np.uint64))
        for m in range(min(100, n_rows - i)):
            keep_p = (1.0 - rates[m % 5]) ** 31
            kept = root[rng.random(root.size) < keep_p]
            fresh = rng.integers(0, 1 << 52, size=4 * num - kept.size + 8, dtype=np.uint64)
            row = np.unique(np.concatenate([kept, fresh]))[:num]
            assert row.size == num
            rows[i] = row
            i += 1
    return rows


# ----------------------------------------------------------------------------------------------
# clocks sampled during the timed regions
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.samples = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self, windows):
        sm, mx, reasons = [], 0, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for t, line in self.samples:
            if not any(a <= t <= b for a, b in windows):
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except (ValueError, IndexError):
                continue
            for nm, val in zip(names, f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------------
# CPU arm: the reference algorithm restated in C (oracle/), all host threads
# ----------------------------------------------------------------------------------------------
def cpu_sketch_rate(reads, n_reads, threads):
    from oracle import oracle as orc
    t0 = time.perf_counter()
    sk = orc.mt_sketch_reads(reads.tobytes() if isinstance(reads, np.ndarray) else reads, n_reads, READ_LEN,
                             list(KSIZES), 0, MAX_HASH_1000, True, threads)
    dt = time.perf_counter() - t0
    return n_reads * READ_LEN / dt / 1e9, dt, sk


def oracle_sketches(rows, num):
    from oracle import oracle as orc
    out = []
    for r in rows:
        o = orc.KmerMinHash(num, 31)
        o.add_many(r)
        out.append(o)
    return out


def cpu_compare_rate(rows, threads):
    """all-vs-all KmerMinHash::compare of the given num=500 rows on `threads` host threads (oracle/baseline_mt.c)"""
    from oracle import oracle as orc
    osk = oracle_sketches(rows, rows.shape[1])
    t0 = time.perf_counter()
    common, size = orc.compare_matrix(osk, osk, nthreads=threads)
    dt = time.perf_counter() - t0
    return len(osk) ** 2 / dt, dt, common, size


def run_reference(args):
    """--impl reference: same metric/config on the host cores.  The Rust crate cannot be built in
    this image (no cargo/rustc), so this is the C restatement of its algorithm (oracle/oracle.c),
    structured like the reference and pinned to its known-answer tests."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    threads = os.cpu_count() or 1
    genome = np_genome(4_000_000, SEED_GENOME)
    calib = np_reads(genome, 1 << 13, SEED_READS)
    _, dt, _ = cpu_sketch_rate(calib, 1 << 13, threads)
    per_step = int(min(1 << 20, max(1 << 13, (1 << 13) * 2.0 / max(dt, 1e-3))))  # about 2 s per step
    batches = [np_reads(genome, per_step, SEED_READS + 1 + b) for b in range(2)]
    for w in range(args.warmup):
        cpu_sketch_rate(batches[w % 2], per_step, threads)
    t0 = time.perf_counter()
    for s in range(args.steps):
        cpu_sketch_rate(batches[s % 2], per_step, threads)
    dt = time.perf_counter() - t0
    value = args.steps * per_step * READ_LEN / dt / 1e9
    # compare half of the metric: a bounded block of cfg3 (BASELINE.md section 3: 2 000 x 2 000 pairs), all host threads
    compare = None
    if not args.no_compare:
        nb = min(args.compare_sketches, 2000)
        rows = planted_sketches(nb, 500, 0x5EED0100)
        c_steps = args.steps
        cpu_compare_rate(rows[:256], threads)
        t0 = time.perf_counter()
        for _ in range(c_steps):
            rate, _, _, _ = cpu_compare_rate(rows, threads)
        dtc = (time.perf_counter() - t0) / c_steps
        compare = {"impl": "reference", "metric": "Jaccard comparisons/s all-vs-all", "value": nb * nb / dtc, "unit": "pairs/s",
                   "ms_per_step": dtc * 1e3, "steps": c_steps, "higher_is_better": True,
                   "config": "cfg3 (num=500, k=31, 100-member clusters): bounded sample, the first %d sketches all-vs-all "
                             "(%d ordered pairs per step), rows spread over %d threads (oracle/baseline_mt.c); time includes "
                             "loading the rows into the CPU sketches" % (nb, nb * nb, threads),
                   "cpu_baseline": {"value": nb * nb / dtc, "unit": "pairs/s", "cores": threads, "kind": "port",
                                    "sample": "%d x %d block of cfg3" % (nb, nb)}}
    line = {
        "impl": "reference", "metric": "Gbp/s sketched", "value": value, "unit": "Gbp/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": "cfg2: scaled=1000 (max_hash=18446744073709552), k=21/31/51 multi-k, 150 bp reads, "
                               "track_abundance; each step a bounded sample of %d reads" % per_step,
                   "reads_per_step": per_step, "read_len": READ_LEN},
        "cpu_baseline": {"value": value, "unit": "Gbp/s", "cores": threads, "kind": "port",
                         "sample": "%d steps x %d reads x 150 bp, 3 k-sizes per base, reads spread over %d threads "
                                   "(oracle/baseline_mt.c)" % (args.steps, per_step, threads)},
        "e2e": {"value": value, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "compare": compare,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(torch, local_rank):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned host buffer is allocated:
    first-touch then places the staging buffers on that node, so that eight ranks feeding eight GPUs do not all pull
    their batches across the socket interconnect.  Best effort: returns the node or None."""
    try:
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        node = int(open("/sys/bus/pci/devices/%s/numa_node" % bdf).read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def run_ours(args):
    import torch
    import torch.distributed as dist
    import sourmash_rust_b200 as smb
    from sourmash_rust_b200 import build
    build.build_library()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this build has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)
    smb.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _, sm_count = smb.device_info()
    lib_stream = torch.cuda.ExternalStream(smb.stream_handle(), device=dev)
    host_threads = max(1, (os.cpu_count() or 1) // world)   # host threads this rank may use

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    R = args.reads_per_step
    n_bytes = R * READ_LEN
    # ---- inputs: same genome on every rank, rank-private read batches (sharded by read batch) ------
    gg = torch.Generator(device=dev)
    gg.manual_seed(SEED_GENOME)
    genome_t = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)[
        torch.randint(0, 4, (GENOME_LEN,), generator=gg, device=dev)]
    n_batches = min(3, args.steps + args.warmup)
    dev_batches = [torch_reads(genome_t, R, SEED_READS + 1000 * rank + b, dev) for b in range(n_batches)]
    host_batches = []
    for b in dev_batches:
        h = torch.empty(n_bytes, dtype=torch.uint8, pin_memory=True)
        h.copy_(b)
        host_batches.append(h)
    torch.cuda.synchronize()

    def new_sketches(ks=KSIZES):
        return [smb.KmerMinHash(0, k, False, 42, MAX_HASH_1000, True) for k in ks]

    clocks = ClockSampler(local_rank)
    clocks.start()
    windows = []
    total_bases = sum_over_ranks(float(args.steps * n_bytes))

    def timed_device(ks):
        """K steps of the batch entry point over device-resident batches; device ms (max over ranks), launches, sketches"""
        mhs = new_sketches(ks)
        for w in range(args.warmup):
            smb.add_reads(mhs, dev_batches[w % n_batches].data_ptr(), R, READ_LEN, force=False, on_device=True)
        for m in mhs:
            m.size()
        mhs = new_sketches(ks)
        barrier()
        launches0 = smb.launch_count()
        t_wall0 = time.time()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(lib_stream)
        for s in range(args.steps):
            smb.add_reads(mhs, dev_batches[s % n_batches].data_ptr(), R, READ_LEN, force=False, on_device=True)
        sizes = [m.size() for m in mhs]  # folds the last candidates into the sorted sketches
        ev1.record(lib_stream)
        barrier()
        windows.append((t_wall0, time.time()))
        return max_over_ranks(ev0.elapsed_time(ev1)), smb.launch_count() - launches0, mhs, sizes

    def timed_e2e(ks):
        """the same K steps from pinned HOST batches through the C ABI, sketches copied back to the host every step"""
        out_m = [torch.zeros(1 << 22, dtype=torch.int64, pin_memory=True) for _ in ks]
        out_a = [torch.zeros(1 << 22, dtype=torch.int64, pin_memory=True) for _ in ks]

        def step(mhs, s):
            smb.add_reads(mhs, host_batches[s % n_batches].data_ptr(), R, READ_LEN, force=False, on_device=False)
            d2h = 0
            for i, m in enumerate(mhs):
                n = smb._call("kmerminhash_copy_mins", m._p, smb._vp(out_m[i].data_ptr()), smb._vp(out_a[i].data_ptr()), False)
                d2h += 16 * n
            return d2h

        warm = new_sketches(ks)
        for w in range(min(args.warmup, 2)):
            step(warm, w)
        mhs = new_sketches(ks)
        barrier()
        t_wall0 = time.time()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(lib_stream)
        d2h_total = 0
        for s in range(args.steps):
            d2h_total += step(mhs, s)
        e1.record(lib_stream)
        barrier()
        windows.append((t_wall0, time.time()))
        return max_over_ranks(e0.elapsed_time(e1)), d2h_total, mhs

    # ---- device-resident path: `value` --------------------------------------------------------------
    ms_dev, launches, mhs, sizes = timed_device(KSIZES)
    # the same K steps once more with per-kernel CUDA events: the three kernels of a step then run
    # one after the other on the library's stream (in the pass above they overlap at their edges on
    # three streams), so that each duration is the kernel's own -- the roofline's denominator
    # (the timed pass uses the fused k=21/31/51 launch; here first the fused kernel alone, then -- with
    # fusion switched off -- one kernel per k-size, so that the k=31 kernel the metric names is measured too)
    smb.profile_enable(True)
    kern = {}
    for fuse, kinds in ((True, ("sketch_multi",)), (False, ("sketch_k21", "sketch_k31", "sketch_k51"))):
        mhs_k = new_sketches()
        smb.fuse_multi_k(fuse)
        for kind in smb.PROFILE_KINDS:
            smb.profile_read(kind, reset=True)
        barrier()
        t_wall0 = time.time()
        for s in range(args.steps):
            smb.add_reads(mhs_k, dev_batches[s % n_batches].data_ptr(), R, READ_LEN, force=False, on_device=True)
        barrier()
        windows.append((t_wall0, time.time()))
        for kind in kinds:
            kern[kind] = smb.profile_read(kind, reset=True)
        del mhs_k
    smb.fuse_multi_k(True)
    smb.profile_enable(False)
    value = total_bases / (ms_dev * 1e-3) / 1e9
    md5_dev = [m.md5sum() for m in mhs]
    outputs = {} if args.dump_outputs and rank == 0 else None
    if outputs is not None:   # the three sketches after the last timed step, as kmerminhash_get_mins / _get_abunds give them
        for k, m in zip(KSIZES, mhs):
            outputs["sketch_k%d_mins" % k] = hash_words(m.mins_np())
            outputs["sketch_k%d_abunds" % k] = m.abunds_np().astype(np.float64)

    # ---- end-to-end path: pinned host buffers in, sketches read back every step ------------------------
    ms_e2e, d2h_total, mhs2 = timed_e2e(KSIZES)
    e2e_value = total_bases / (ms_e2e * 1e-3) / 1e9
    assert [m.md5sum() for m in mhs2] == md5_dev, "device-resident and host-fed paths disagree"
    abunds_dev = [m.abunds_np() for m in mhs]

    # ---- the BASELINE metric's literal configuration: ONE sketch, k=31, scaled=1000 -------------------------
    ms_k31, launches_k31, mhs_k31, sizes_k31 = timed_device((31,))
    ms_k31_e2e, d2h_k31, mhs_k31_h = timed_e2e((31,))
    assert mhs_k31_h[0].md5sum() == mhs_k31[0].md5sum() == md5_dev[1]
    k31 = {"metric": "Gbp/s sketched (k=31, scaled=1000)", "value": total_bases / (ms_k31 * 1e-3) / 1e9, "unit": "Gbp/s",
           "ms_per_step": ms_k31 / args.steps, "gpu_launches": launches_k31,
           "e2e": {"value": total_bases / (ms_k31_e2e * 1e-3) / 1e9, "unit": "Gbp/s", "ms_per_step": ms_k31_e2e / args.steps,
                   "h2d_bytes_per_step": n_bytes, "d2h_bytes_per_step": d2h_k31 // max(1, args.steps)},
           "config": "one KmerMinHash(num=0, k=31, max_hash=18446744073709552, track_abundance) through kmerminhash_add_reads, "
                     "same read batches as the multi-k run"}

    # ---- what the host side can deliver at most: bare pinned-host -> device copies, all ranks at once ---------------------
    h2d_dst = torch.empty(n_bytes, dtype=torch.uint8, device=dev)
    cp_stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(cp_stream):
        h2d_dst.copy_(host_batches[0], non_blocking=True)
    barrier()
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 4
    with torch.cuda.stream(cp_stream):
        c0.record(cp_stream)
        for i in range(reps):
            h2d_dst.copy_(host_batches[i % n_batches], non_blocking=True)
        c1.record(cp_stream)
    barrier()
    h2d_gbs = n_bytes * reps / (max_over_ranks(c0.elapsed_time(c1)) * 1e-3) / 1e9   # per GPU, slowest rank
    del h2d_dst

    # ---- NOT a reference format: the same reads 2 bits per base from pinned host memory (a quarter of the PCIe bytes) ----
    packed = None
    if not args.no_packed:
        packed_batches = []
        for hb in host_batches:
            pk = smb.pack_2bit(hb.numpy().reshape(R, READ_LEN), READ_LEN)
            t = torch.empty(pk.size, dtype=torch.uint8, pin_memory=True)
            t.copy_(torch.from_numpy(pk.reshape(-1)))
            packed_batches.append(t)
        out_m = [torch.zeros(1 << 22, dtype=torch.int64, pin_memory=True) for _ in KSIZES]
        out_a = [torch.zeros(1 << 22, dtype=torch.int64, pin_memory=True) for _ in KSIZES]

        def p_step(sk, s):
            smb.add_reads_2bit(sk, packed_batches[s % n_batches].data_ptr(), R, READ_LEN)
            for i, m in enumerate(sk):
                smb._call("kmerminhash_copy_mins", m._p, smb._vp(out_m[i].data_ptr()), smb._vp(out_a[i].data_ptr()), False)

        warm = new_sketches()
        for w in range(2):
            p_step(warm, w)
        pm = new_sketches()
        barrier()
        t_wall0 = time.time()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(lib_stream)
        for s in range(args.steps):
            p_step(pm, s)
        e1.record(lib_stream)
        barrier()
        windows.append((t_wall0, time.time()))
        ms_p = max_over_ranks(e0.elapsed_time(e1))
        assert [m.md5sum() for m in pm] == md5_dev, "2-bit input and ASCII input disagree"
        packed = {"value": total_bases / (ms_p * 1e-3) / 1e9, "unit": "Gbp/s", "ms_per_step": ms_p / args.steps,
                  "h2d_bytes_per_step": int(packed_batches[0].numel()),
                  "entry_point": "kmerminhash_add_reads_2bit (include/sourmash_b200.h): NOT a reference input format -- reads 2 bits "
                                 "per base in pinned host memory, expanded to ASCII on the device behind the copy; same sketches "
                                 "(md5 asserted)", "parity_with_ascii_path": True}
        del packed_batches, pm, warm

    # ---- the reference's own calling pattern: one kmerminhash_add_sequence call per read and per k-size ---------
    # (src/ffi.rs:55-70; a C loop over the unmodified symbol, sourmash_rust_b200/host/feed_reads.c).  Reads as
    # NUL-terminated strings in host memory; T host threads, each feeding its own three sketches with its share of
    # the batch; the timed region ends when every sketch has been flushed; the threads' sketches are then merged.
    percall = None
    if not args.no_percall:
        T = max(1, min(args.percall_threads or 4, host_threads))
        z = np.zeros((R, READ_LEN + 1), dtype=np.uint8)
        z[:, :READ_LEN] = host_batches[0].numpy().reshape(R, READ_LEN)
        pc_steps = args.steps
        warm_reads = min(R // T // 8, 50_000)
        secs, groups = 0.0, None
        barrier()
        t_wall0 = time.time()
        for s in range(pc_steps):
            groups = [new_sketches() for _ in range(T)]
            secs += smb.feed_reads(groups, z, R, READ_LEN + 1, force=False, warm_reads=warm_reads)
        windows.append((t_wall0, time.time()))
        timed_reads = R - warm_reads * T
        secs = max_over_ranks(secs)
        # parity: thread sketches merged == the batch entry point over the same reads
        merged = groups[0]
        for g in groups[1:]:
            for a, b in zip(merged, g):
                a.merge(b)
        chk = new_sketches()
        smb.add_reads(chk, host_batches[0].data_ptr(), R, READ_LEN, force=False, on_device=False)
        for a, b in zip(merged, chk):
            assert a.md5sum() == b.md5sum() and np.array_equal(a.abunds_np(), b.abunds_np()), "per-call path differs from the batch path"
        percall = {"value": sum_over_ranks(float(pc_steps * timed_reads * READ_LEN)) / secs / 1e9, "unit": "Gbp/s",
                   "entry_point": "kmerminhash_add_sequence (include/sourmash.h), one call per read and per k-size",
                   "host_threads_per_gpu": T, "calls_per_step": timed_reads * len(KSIZES),
                   "ns_per_call_per_thread": secs / (pc_steps * timed_reads * len(KSIZES)) * T * 1e9,
                   "ms_per_step": secs / pc_steps * 1e3, "h2d_bytes_per_step": timed_reads * READ_LEN * len(KSIZES),
                   "parity_with_batch_path": True,
                   "note": "host-bound: each call validates and stages its read on the host (deferred, flushed in 8 MiB "
                           "batches per sketch); round 1 went to the device on every call: 45 us per call = 0.003 Gbp/s"}
        del z, groups, merged, chk

    # ---- roofline of the dominant kernel (the fused k=21/31/51 launch; k=31 is the metric's k) ---
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except (OSError, ValueError):
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
    consts = kernel_constants()
    k31_ms, k31_n = kern["sketch_k31"]
    km_ms, km_n = kern["sketch_multi"]
    per_k = {}
    for k, kind in zip(KSIZES + ("multi",), ("sketch_k21", "sketch_k31", "sketch_k51", "sketch_multi")):
        ms, n = kern[kind]
        if n:
            per_k["k%s" % k] = {"launches": n, "avg_ms": ms / n, "gbp_s": args.steps * n_bytes / (ms * 1e-3) / 1e9}

    # ---- all-vs-all compare (cfg3), rows sharded by rank, CSR all-gathered over NCCL inside the library -------------
    compare = None
    if not args.no_compare:
        compare = bench_compare(args, smb, torch, dist, dev, rank, world, barrier, max_over_ranks, lib_stream, windows,
                                host_threads, hbm_peak, peak_src, outputs)

    clocks.stop()

    # ---- CPU baseline next to it (rank 0, N=1 only): bounded sample of the same workload --------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from oracle import oracle as orc
        orc.build()
        threads = os.cpu_count() or 1
        sample_reads = host_batches[0].numpy()
        _, dt, _ = cpu_sketch_rate(sample_reads[: (1 << 13) * READ_LEN], 1 << 13, threads)
        n_s = int(min(R, max(1 << 13, (1 << 13) * 12.0 / max(dt, 1e-3))))
        rate, dt, osk = cpu_sketch_rate(sample_reads[: n_s * READ_LEN], n_s, threads)
        cpu = {"value": rate, "unit": "Gbp/s", "cores": threads, "kind": "port",
               "sample": "first %d reads of batch 0 (%.1f s on %d threads), 3 k-sizes per base" % (n_s, dt, threads)}
        # the same sample through the GPU path must give the same sketches
        chk = new_sketches()
        smb.add_reads(chk, host_batches[0].data_ptr(), n_s, READ_LEN, force=False, on_device=False)
        for g, o in zip(chk, osk):
            assert g.md5sum() == o.md5sum() and np.array_equal(g.abunds_np(), o.abunds_np()), "GPU/CPU sketches differ"
        cpu["parity_checked"] = True

    clk = clocks.summary(windows)
    roof = roof_hbm = None
    if rank == 0 and km_n:
        # The binding roof of the sketch kernels is integer issue, not HBM (three MurmurHash3 per byte read).  Two
        # readings: (1) issue slots -- 4 warp instructions per clock per SM at the SM clock seen during the run, with the
        # executed instruction count per window from the ncu capture; (2) the hash-only ceiling -- MurmurHash3 of
        # register-resident k-mers and nothing else, measured live (smgpu_int_peak modes 10-12).
        kc = consts.get(KERNEL_OF["multi"], {})
        kc31 = consts.get(KERNEL_OF[31], {})
        mhz = clk.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
        issue_peak = 4 * 32 * sm_count * mhz * 1e6
        windows_per_launch = args.steps * n_bytes / km_n
        launch_s = km_ms / km_n * 1e-3
        hash_rate = {k: smb.int_peak(mode, 256, sm_count * 8) for mode, k in ((10, 21), (11, 31), (12, 51))}
        ceiling = 1.0 / sum(1.0 / hash_rate[k] for k in KSIZES)  # windows/s if the three hashes were all there is
        achieved_w = windows_per_launch / launch_s
        ipw = kc.get("instr_per_unit")
        roof = {"bound": "int_issue", "kernel": KERNEL_OF["multi"],
                "achieved": ipw * achieved_w / 1e12 if ipw else None, "peak": issue_peak / 1e12, "unit": "Tinstr/s",
                "frac": ipw * achieved_w / issue_peak if ipw else None,
                "traffic": kc.get("dram_bytes_per_unit") * windows_per_launch if kc.get("dram_bytes_per_unit") else None,
                "instr_per_window": ipw, "windows_per_launch": windows_per_launch, "avg_launch_ms": km_ms / km_n,
                "peak_source": "4 warp-instr/clk/SM x 32 lanes x %d SMs x %.0f MHz (SM clock sampled during the run)" % (sm_count, mhz),
                "constants_source": kc.get("source"),
                "ncu": {"issue_slots_pct": kc.get("issue_pct"), "alu_pipe_pct": kc.get("alu_pct"), "fmaheavy_pipe_pct": kc.get("fmaheavy_pct")},
                "duration_source": "CUDA events around each launch on the library's stream, separate pass of the same K steps",
                "hash_only_ceiling": {"g_hashes_s": {"k%d" % k: hash_rate[k] / 1e9 for k in KSIZES},
                                      "fused_gbp_s": ceiling / 1e9, "frac": achieved_w / ceiling,
                                      "how": "MurmurHash3 x64_128 of register-resident k-mers, no staging / strand "
                                             "choice / shared memory (hash_peak_kernel), measured in this run"},
                "k31_kernel": {"gbp_s": args.steps * n_bytes / (k31_ms * 1e-3) / 1e9 if k31_n else None,
                               "instr_per_window": kc31.get("instr_per_unit"),
                               "issue_frac": (kc31["instr_per_unit"] * (args.steps * n_bytes) / (k31_ms * 1e-3) / issue_peak)
                               if k31_n and kc31.get("instr_per_unit") else None,
                               "hash_only_frac": (args.steps * n_bytes / (k31_ms * 1e-3) / hash_rate[31]) if k31_n else None},
                "note": "binding resource of the sketch kernels: ALU + FMA-heavy (IMAD) pipes; HBM side in roofline_hbm"}
        achieved_gbs = windows_per_launch / launch_s / 1e9   # 1 B (one ASCII base) per window start, SURVEY 8(d)
        roof_hbm = {"bound": "hbm", "kernel": KERNEL_OF["multi"], "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s",
                    "frac": achieved_gbs / hbm_peak, "traffic": roof["traffic"], "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": windows_per_launch,
                    "note": "not the binding resource: the kernel reads each base once (ncu DRAM bytes per window in `traffic`)"}
    if rank == 0:
        line = {
            "metric": "Gbp/s sketched", "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_dev / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": {"workload": "cfg2: scaled=1000 (max_hash=18446744073709552), k=21/31/51 multi-k, 150 bp reads, "
                                   "track_abundance, %d reads (%d MB ASCII) per step per GPU" % (R, n_bytes >> 20),
                       "reads_per_step_per_gpu": R, "read_len": READ_LEN, "sharding": "read batches per rank, no collective",
                       "l2": "inputs (%d MB per step) larger than the 126 MB L2; %d distinct batches cycled" % (n_bytes >> 20, n_batches),
                       "sketch_sizes": sizes, "host_numa_node": numa},
            "e2e": {"value": e2e_value, "unit": "Gbp/s", "h2d_bytes_per_step": n_bytes,
                    "d2h_bytes_per_step": d2h_total // max(1, args.steps), "ms_per_step": ms_e2e / args.steps,
                    "entry_point": "kmerminhash_add_reads (batch extension, include/sourmash_b200.h), pinned host buffers",
                    "h2d_ceiling_gbs": h2d_gbs,
                    "h2d_ceiling_note": "bare cudaMemcpyAsync of the same pinned batches, all ranks at once, per GPU (slowest "
                                        "rank): what the host side can deliver; 1 B per base, so this is also the e2e "
                                        "ceiling in Gbp/s per GPU",
                    "frac_of_h2d_ceiling": (e2e_value / world) / h2d_gbs},
            "e2e_per_call": percall,
            "e2e_packed_2bit": packed,
            "k31_scaled1000": k31,
            "gpu_launches": launches,
            "roofline": roof, "roofline_hbm": roof_hbm, "sketch_kernels": per_k,
            "cpu_baseline": cpu,
            "clocks": clk,
            "compare": compare,
        }
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def bench_compare(args, smb, torch, dist, dev, rank, world, barrier, max_over_ranks, lib_stream, windows, host_threads,
                  hbm_peak, peak_src, outputs):
    N, NUM = args.compare_sketches, 500
    rows = planted_sketches(N, NUM, 0x5EED0100)
    from sourmash_rust_b200 import sharding
    r0, r1 = sharding.shard_range(N, rank, world)
    nr = r1 - r0
    # the library's own communicator (NCCL inside libsourmash.so); the id travels over the host program's channel
    if world > 1:
        smb.comm_init_from_torch()   # (one rank: no communicator needed, the collectives act as a world of one)
    # this rank's sketches: a resident collection (rows checked sorted once, here); the step gathers and compares
    local = smb.SketchCollection.from_csr(rows[r0:r1].reshape(-1), np.arange(nr + 1, dtype=np.uint64) * np.uint64(NUM),
                                          nr, NUM, 31, 42, 0)
    common = torch.empty((max(1, nr), N), dtype=torch.int32, device=dev)
    size = torch.empty((max(1, nr), N), dtype=torch.int32, device=dev)
    ratio = torch.empty((max(1, nr), N), dtype=torch.float64, device=dev)
    steps = args.steps

    def step():
        # all-gather of the packed sketches over NCCL/NVLink + this rank's row block, in one library call: the
        # join's hash table over the rank's own rows is built while the other ranks' rows are in flight
        return smb.compare_matrix_allgather_device(local, "compare", common.data_ptr(), size.data_ptr(), ratio.data_ptr(), N)

    for _ in range(3):
        step()
    smb.profile_enable(True)
    for kind in smb.PROFILE_KINDS:
        smb.profile_read(kind, reset=True)
    barrier()
    t_wall0 = time.time()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lib_stream)
    for _ in range(steps):
        step()
    e1.record(lib_stream)
    barrier()
    windows.append((t_wall0, time.time()))
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    kern = {kind: smb.profile_read(kind, reset=True) for kind in smb.PROFILE_KINDS if kind.startswith(("compare", "join"))}
    smb.profile_enable(False)

    # ---- parity on every rank: 10^6 sampled pairs of this rank's block against the oracle (SURVEY 8(d) cfg3) -------------
    from oracle import oracle as orc
    osk = oracle_sketches(rows, NUM)
    rng = np.random.Generator(np.random.PCG64(77 + rank))
    n_s = args.compare_samples
    ii = rng.integers(0, max(1, nr), size=n_s)
    jj = rng.integers(0, N, size=n_s)
    rel = rng.random(n_s) < 0.5                      # half of the samples inside the row's own 100-member cluster (related pairs)
    jj[rel] = ((r0 + ii[rel]) // 100) * 100 + rng.integers(0, 100, size=int(rel.sum()))
    jj = np.minimum(jj, N - 1)
    oc, osz = orc.compare_pairs(osk, r0 + ii, jj, nthreads=host_threads)
    ti, tj = torch.from_numpy(ii).to(dev), torch.from_numpy(jj).to(dev)
    gc, gs, gr = common[ti, tj].cpu().numpy(), size[ti, tj].cpu().numpy(), ratio[ti, tj].cpu().numpy()
    ok = bool(np.array_equal(gc.astype(np.uint32), oc) and np.array_equal(gs.astype(np.uint32), osz) and
              np.array_equal(gr, oc.astype(np.float64) / np.maximum(1, osz).astype(np.float64)))
    assert ok, "rank %d: sampled pairs differ from the oracle" % rank
    nonzero = int((oc > 0).sum())
    if outputs is not None:   # the last timed step's matrix at (a prefix of) the seeded sample of cells just checked
        m = min(n_s, DUMP_COMPARE_CELLS)
        outputs.update(compare_rows=(r0 + ii[:m]).astype(np.float64), compare_cols=jj[:m].astype(np.float64),
                       compare_common=gc[:m].astype(np.float32), compare_size=gs[:m].astype(np.float32),
                       compare_ratio=gr[:m].astype(np.float64))

    # ---- the same matrix with the data-driven path choice overridden: every pair walked (dense kernel) --------------------
    smb.compare_path("dense")
    step()
    barrier()
    e0.record(lib_stream)
    for _ in range(steps):
        step()
    e1.record(lib_stream)
    barrier()
    ms_dense = max_over_ranks(e0.elapsed_time(e1)) / steps
    smb.compare_path("auto")

    # ---- end to end: host CSR in, f64 Jaccard matrix out to pinned host memory ----------------------------------------------
    out = torch.empty((max(1, nr), N), dtype=torch.float64, pin_memory=True)
    rows_pin = torch.from_numpy(np.ascontiguousarray(rows[r0:r1]).view(np.int64).reshape(-1)).pin_memory()
    offs_pin = torch.from_numpy((np.arange(nr + 1, dtype=np.uint64) * np.uint64(NUM)).view(np.int64)).pin_memory()
    rows_c, offs_c = rows_pin.numpy().view(np.uint64), offs_pin.numpy().view(np.uint64)

    def e2e():
        # this rank's sketches from host memory (upload + sortedness check), gather, row block, matrix back to the host
        loc = smb.SketchCollection.from_csr(rows_c, offs_c, nr, NUM, 31, 42, 0, on_device=False)
        smb.SketchCollection(_ptr=smb._call("smgpu_compare_matrix_allgather", loc._p, 0, None, None, smb._vp(out.data_ptr()), N, False))

    e2e()
    barrier()
    e0.record(lib_stream)
    for _ in range(steps):
        e2e()
    e1.record(lib_stream)
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1)) / steps
    assert np.array_equal(out[:4].numpy(), ratio[:4].cpu().numpy())

    # ---- CPU baseline of the compare half (rank 0, N=1 only): bounded block, all host threads --------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        nb = min(N, 2000)
        rate, dt, oc2, osz2 = cpu_compare_rate(rows[:nb], os.cpu_count() or 1)
        assert np.array_equal(common[:nb, :nb].cpu().numpy().astype(np.uint32), oc2), "compare matrix differs from the CPU block"
        cpu = {"value": rate, "unit": "pairs/s", "cores": os.cpu_count() or 1, "kind": "port",
               "sample": "the first %d x %d block of the matrix (%.2f s on %d threads), three-pass KmerMinHash::compare per pair "
                         "(oracle/baseline_mt.c)" % (nb, nb, dt, os.cpu_count() or 1), "parity_checked": True}
    smb.comm_destroy()

    pairs = float(N) * float(N)
    out_bytes = 16.0 * pairs / world     # u32 common + u32 size + f64 ratio per cell of this rank's block
    kms = {k: (v[0] / steps) for k, v in kern.items() if v[1]}
    return {"metric": "Jaccard comparisons/s all-vs-all", "value": pairs / (ms * 1e-3), "unit": "pairs/s",
            "config": "cfg3: %d sketches, num=500, k=31, 100 clusters of 100 (1 %% of the pairs related), full ordered matrix "
                      "(common,size u32 + Jaccard f64), rows sharded over %d rank(s); each step = all-gather of the packed "
                      "sketches over NCCL inside the library + this rank's row block (smgpu_compare_matrix_allgather)" % (N, world),
            "ms_per_step": ms, "steps": steps, "scaling": "strong",
            "kernel_ms_per_step": kms,
            "e2e": {"value": pairs / (ms_e2e * 1e-3), "unit": "pairs/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int(rows_c.nbytes + offs_c.nbytes),
                    "d2h_bytes_per_step": int(nr * N * 8)},
            "path": "auto: hash-grouped inverted-index join finds the related pairs (here 1 % of all: the figure is data-dependent), "
                    "only those are walked; every-pair figure in dense_path",
            "dense_path": {"value": pairs / (ms_dense * 1e-3), "unit": "pairs/s", "ms_per_step": ms_dense,
                           "note": "every pair walked: rank-compressed fixed-length walk, smgpu_compare_path(1)"},
            "roofline": {"bound": "hbm", "kernel": "whole matrix step (join + fill_cells + walk_pairs)",
                         "achieved": out_bytes / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": out_bytes / (ms * 1e-3) / 1e9 / hbm_peak, "traffic": None, "peak_source": peak_src,
                         "algorithmic_bytes_per_step": out_bytes,
                         "note": "compulsory HBM traffic of a row block is its 16 B per cell of output; the step is bound by "
                                 "integer issue and latency in the join and the pair walk, not by HBM (profiles/)"},
            "cpu_baseline": cpu,
            "operand_bytes_per_pair": 2 * NUM * 8,
            "parity": {"sampled_pairs_per_rank": int(n_s), "related_samples": nonzero, "ranks_checked": world, "ok": ok}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads-per-step", type=int, default=1 << 21)
    ap.add_argument("--compare-sketches", type=int, default=10000)
    ap.add_argument("--compare-samples", type=int, default=1_000_000)
    ap.add_argument("--percall-threads", type=int, default=0)
    ap.add_argument("--no-compare", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-percall", action="store_true")
    ap.add_argument("--no-packed", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write, as DIR/<name>.npy (float32/float64), what the timed paths computed in "
                         "their last step: the three sketches' hashes (high and low 32 bits) and abundances, and the "
                         "compare matrix at a seeded sample of cells")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
