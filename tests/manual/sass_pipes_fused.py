"""Static pipe model of the sketch kernels' k-mer loops, for builds whose multi-k kernels run one fused loop:
`python tests/manual/sass_pipes_fused.py [LIB.so | KERNEL.cubin]` (default: sourmash_rust_b200/libsourmash.so).

Same parsing, costs and assumptions as tests/manual/sass_pipes.py, which expects one k-mer loop per k-size.  Here a
`sketch_kernel<KA,KB,KC>` may instead hold ONE loop whose trip handles a window start for every k-size of the launch
(kmer_loop_fused): it then has one survivor path per k-size and window start, and its row -- labelled `k21+31+51` --
is the whole loop per warp and window start.  Single-k kernels, and builds with one loop per k-size, read as in
sass_pipes.py.
"""
import collections
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sass_pipes import ROOT, cost, kernel_ks, kmer_loops, loop_body, parse  # noqa: E402

KEYS = ("issue", "fma", "alu", "lsu", "wide", "wide_acc")


def model(path):
    """{"KA,KB,KC": {"k21+31+51" or "k21", ...: {...}, "total": {...}}} per warp and window start"""
    res = {}
    for name, ins in sorted(parse(path).items(), key=lambda kv: kernel_ks(kv[0])):
        ks = kernel_ks(name)
        loops = kmer_loops(ins)
        if len(loops) == len(ks):
            groups = [[k] for k in ks]
        elif len(loops) == 1:
            groups = [ks]
        else:
            raise SystemExit("%s: found %d k-mer loops for k = %s" % (name, len(loops), ks))
        row, tot = {}, collections.Counter()
        for g, (first, last) in zip(groups, loops):
            label = "k" + "+".join(str(k) for k in g)
            body, n_surv = loop_body(ins, first, last)
            if n_surv == 0 or n_surv % len(g):
                raise SystemExit("%s: %d survivor paths in the %s loop" % (name, n_surv, label))
            windows = n_surv // len(g)  # window starts per trip
            c = cost(body)
            row[label] = {key: c[key] / windows for key in KEYS}
            row[label]["windows_per_trip"] = windows
            for key in KEYS:
                tot[key] += c[key] / windows
        row["total"] = dict(tot)
        res[",".join(str(k) for k in ks + [0] * (3 - len(ks)))] = row
    return res


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "sourmash_rust_b200", "libsourmash.so")
    print("per warp and window start (cycles; issue in slots); FMA = FMA-heavy pipe; wide+acc = IMAD.WIDE with a "
          "register addend")
    print("%-24s %-10s %7s %7s %7s %6s %7s %9s" % ("kernel", "loop", "issue", "FMA", "ALU", "LSU", "max", "wide+acc"))
    for kern, row in model(path).items():
        for loop, c in row.items():
            print("%-24s %-10s %7.1f %7.1f %7.1f %6.1f %7.1f %9.1f" % (
                "sketch_kernel<%s>" % kern, loop, c["issue"], c["fma"], c["alu"], c["lsu"],
                max(c["issue"], c["fma"], c["alu"]), c["wide_acc"]))


if __name__ == "__main__":
    main()
