"""Static pipe model of the sketch kernels' k-mer loops, from the SASS of the built library (no GPU needed):
`python tests/manual/sass_pipes.py [LIB.so | KERNEL.cubin]` (default: sourmash_rust_b200/libsourmash.so).

For every `sketch_kernel<KA,KB,KC>` it finds one k-mer loop per k-size, leaves out the survivor path, and prints per
warp and window start (one window per lane) the issue slots and the cycles each integer pipe is held, and the max of
those three.  On the B200 the kernels' time has followed the issue-slot count, not the FMA-heavy figure
(profiles/sketch_pipes_r3.md, DESIGN 4.1); the pipe figures show how far each pipe sits below issue.

Assumptions (pipe costs from profiles/intpeak_r2.md, a B200 sub-partition):
  * issue: one slot per SASS instruction, whatever its pipe;
  * FMA-heavy pipe: IMAD / IMAD.MOV / IMAD.IADD / IMAD.SHL / IMAD.X / IMAD.U32 2 cycles; IMAD.HI and IMAD.WIDE with an RZ
    addend 4; IMAD.WIDE with a register-pair addend (the 64-bit accumulating form) 8;
  * ALU pipe, 2 cycles each: LOP3, SHF, IADD3, LEA, ISETP, SEL, PRMT, PLOP3, FLO, BREV, POPC, IABS, IMNMX, MOV, and VIADD
    (counted as ALU, though ptxas may also place it on the FMA-heavy pipe);
  * LSU: shared-memory bandwidth, 1 cycle per 32-bit warp access (LDS 1, LDS.64 2, LDS.128 4, same for STS);
  * everything else (branches, BSSY / BSYNC, uniform-datapath U* instructions, NOP) takes an issue slot only;
  * a loop trip handles one window per lane for each survivor path it contains; the survivor path (a forward branch
    over the code that writes a survivor with a global atomic or store) is rare and is left out, and so are
    out-of-line divergence paths that sit after the function's EXIT.
Stalls, dual-issue limits and instruction-cache misses are not modelled.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")

ALU = {"LOP3", "SHF", "IADD3", "LEA", "ISETP", "SEL", "PRMT", "PLOP3", "FLO", "BREV", "POPC", "IABS", "IMNMX", "MOV",
       "VIADD"}
LSU = {"LDS", "STS"}
GLOBAL_WRITE = ("ATOMG", "ATOM", "RED", "STG", "ST")


def parse(path):
    """{mangled kernel name: [(address, instruction text)]} for every sketch_kernel in the file"""
    sass = subprocess.run([CUOBJDUMP, "-sass", path], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                          check=True).stdout
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1) if "sketch_kernel" in m.group(1) else None
            if cur:
                funcs[cur] = []
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if cur and m:
            funcs[cur].append((int(m.group(1), 16), m.group(2)))
    return funcs


def opcode(text):
    return re.sub(r"^@!?U?P\w+\s+", "", text).split()[0]


def branch_target(text):
    m = re.match(r"(?:@!?U?P\w+\s+)?BRA(?:\.\S+)?\s+(?:!?U?P\w+,\s*)?(0x[0-9a-f]+)", text)
    return int(m.group(1), 16) if m else None


def kmer_loops(ins):
    """[(first, last) index] of the k-mer loops, in program order: the backward branches whose body holds the
    survivor path (a forward branch over a global atomic) and MurmurHash3's c1 constant"""
    idx = {a: i for i, (a, _) in enumerate(ins)}
    last_exit = max(i for i, (_, t) in enumerate(ins) if opcode(t) == "EXIT")
    loops = []
    for i, (a, t) in enumerate(ins[:last_exit]):  # past the last EXIT: out-of-line paths that jump back, not loops
        tgt = branch_target(t)
        if tgt is None or tgt >= a or tgt not in idx:
            continue
        body = ins[idx[tgt]:i + 1]
        if any("0x114253d5" in x for _, x in body) and any(opcode(x).startswith("ATOMG") for _, x in body):
            loops.append((idx[tgt], i))
    # keep the innermost: drop a loop that contains another one found
    inner = [l for l in loops if not any(o != l and l[0] <= o[0] and o[1] <= l[1] for o in loops)]
    return sorted(inner)


def loop_body(ins, first, last):
    """the loop's instructions without its survivor paths; returns (instructions, number of survivor paths)"""
    out, n_surv, skip_to = [], 0, None
    for i in range(first, last + 1):
        a, t = ins[i]
        if skip_to is not None:
            if a < skip_to:
                continue
            skip_to = None
        tgt = branch_target(t)
        if tgt is not None and a < tgt <= ins[last][0]:
            skipped = [x for b, x in ins[i + 1:last + 1] if b < tgt]
            writes = [j for j, x in enumerate(skipped) if opcode(x).split(".")[0] in GLOBAL_WRITE]
            # the survivor path starts at the first such branch after the hash's last wide multiply (an earlier one,
            # such as a branch over an invalid window's whole hash, skips common-path work and is counted not taken)
            hashing = writes and any(opcode(x).startswith("IMAD.WIDE") for x in skipped[:writes[0]])
            if writes and not hashing:
                out.append(t)
                n_surv += 1
                skip_to = tgt
                continue
        out.append(t)
    return out, n_surv


def cost(body):
    c = collections.Counter()
    for t in body:
        op = opcode(t)
        base = op.split(".")[0]
        c["issue"] += 1
        if base == "IMAD":
            if ".WIDE" in op:
                acc = t.split(",")[-1].strip() != "RZ"
                c["fma"] += 8 if acc else 4
                c["wide_acc" if acc else "wide"] += 1
            elif ".HI" in op:
                c["fma"] += 4
            else:
                c["fma"] += 2
        elif base in ALU:
            c["alu"] += 2
        elif base in LSU:
            c["lsu"] += 4 if ".128" in op else 2 if ".64" in op else 1
    return c


def kernel_ks(name):
    m = re.search(r"sketch_kernelILi(\d+)ELi(\d+)ELi(\d+)E", name)
    return [int(k) for k in m.groups() if int(k)] if m else []


def model(path):
    """{"KA,KB,KC": {"k21": {...}, ..., "total": {...}}} per warp-window"""
    res = {}
    for name, ins in sorted(parse(path).items(), key=lambda kv: kernel_ks(kv[0])):
        ks = kernel_ks(name)
        loops = kmer_loops(ins)
        if len(loops) != len(ks):
            raise SystemExit("%s: found %d k-mer loops for k = %s" % (name, len(loops), ks))
        row, tot = {}, collections.Counter()
        for k, (first, last) in zip(ks, loops):
            body, n_surv = loop_body(ins, first, last)
            if n_surv == 0:
                raise SystemExit("%s: no survivor path found in the k=%d loop" % (name, k))
            c = cost(body)
            row["k%d" % k] = {key: c[key] / n_surv for key in ("issue", "fma", "alu", "lsu", "wide", "wide_acc")}
            row["k%d" % k]["windows_per_trip"] = n_surv
            for key in ("issue", "fma", "alu", "lsu", "wide", "wide_acc"):
                tot[key] += c[key] / n_surv
        row["total"] = dict(tot)
        res[",".join(str(k) for k in kernel_ks(name) + [0] * (3 - len(ks)))] = row
    return res


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "sourmash_rust_b200", "libsourmash.so")
    print("per warp and window start (cycles; issue in slots); FMA = FMA-heavy pipe; wide+acc = IMAD.WIDE with a "
          "register addend")
    print("%-24s %-6s %7s %7s %7s %6s %7s %9s" % ("kernel", "loop", "issue", "FMA", "ALU", "LSU", "max", "wide+acc"))
    for kern, row in model(path).items():
        for loop, c in row.items():
            print("%-24s %-6s %7.1f %7.1f %7.1f %6.1f %7.1f %9.1f" % (
                "sketch_kernel<%s>" % kern, loop, c["issue"], c["fma"], c["alu"], c["lsu"],
                max(c["issue"], c["fma"], c["alu"]), c["wide_acc"]))


if __name__ == "__main__":
    main()
