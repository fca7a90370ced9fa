"""Read classes and the abundance EM (Hansel.read_classes, em_abundance) on config 3: 10M x 150 bp reads over N = 10k
sites, against haplotypes that are the 5 strains plus random mutants of them, for H in {5, 50, 100}; and the ONT
workload at H = 50.

Per H: the class kernels' device time (hx_last_kernel_ms(5), best of --reps after a warm-up call) next to the
assignment kernels' (hx_last_kernel_ms(3)) on the same input, the tied reads (the assigned reads outside singleton
classes) and the classes, the EM's host time and iterations, and the wall time of read_classes from host arrays.
The oracle (oracle/abundance_oracle.py) checks the classes on a subsample and the first 50 EM iterations bit
for bit.  Card name and power limit are read in the same run.  One JSON line per measurement; --out also writes
them to a file.

    python tools/abundance_bench.py [--reps 10] [--out results/abundance_bench.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gretel_b200 import synth  # noqa: E402
from gretel_b200.hansel import REF_SYMBOLS, REF_UNSYMBOLS, Hansel, em_abundance  # noqa: E402
from oracle import abundance_oracle as ao  # noqa: E402
from support_bench import card, haplotypes  # noqa: E402


def measure(name, d, N, Hs, reps, check_reads, emit):
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=1, device=0)
    rank, off, codes = d["rank"], d["off"], d["codes"]
    R = len(rank)
    for H in Hs:
        haps = haplotypes(d["strains"], H)
        h.assign_reads(haps, rank, off, codes)                       # warm-up
        assign = []
        for _ in range(reps):
            h.assign_reads(haps, rank, off, codes)
            assign.append(h.kernel_ms("assign"))
        cls = h.read_classes(haps, rank, off, codes)                 # warm-up
        kern, wall = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            cls = h.read_classes(haps, rank, off, codes)
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(h.kernel_ms("classes"))
        em_ms = []
        for _ in range(max(3, reps // 2)):
            t0 = time.perf_counter()
            em = em_abundance(H, cls)
            em_ms.append((time.perf_counter() - t0) * 1e3)
        # the Python EM is slow: it checks the first 50 iterations, bit for bit
        exp, em50 = ao.em(H, cls.class_off, cls.members, cls.count, max_iter=50), em_abundance(H, cls, max_iter=50)
        em_equal = (em50.pi.tobytes() == np.array(exp["pi"]).tobytes() and em50.n_iter == exp["n_iter"]
                    and em50.loglik == exp["loglik"])
        n = min(R, check_reads)
        sub = h.read_classes(haps, rank[:n], off[:n + 1], codes)
        ref = ao.classes(haps, rank[:n], off[:n + 1], codes)
        cls_equal = all(np.array_equal(getattr(sub, k), ref[k]) for k in ("class_off", "members", "count"))
        size = np.diff(cls.class_off)
        emit({"workload": name, "reads": R, "H": H, "classes_kernel_ms": min(kern),
              "classes_kernel_ms_median": float(np.median(kern)), "assign_kernel_ms": min(assign),
              "classes_over_assign": min(kern) / min(assign), "read_classes_wall_ms": min(wall),
              "read_classes_wall_ms_median": float(np.median(wall)), "assigned": cls.assigned,
              "tied_reads": int(cls.count[size >= 2].sum()), "classes": len(cls),
              "tied_classes": int((size >= 2).sum()), "em_ms": min(em_ms), "em_iterations": em.n_iter,
              "em_converged": em.converged, "oracle_reads": n, "oracle_classes_equal": cls_equal,
              "oracle_em_equal": em_equal})
        if not (cls_equal and em_equal):
            raise SystemExit("classes or EM differ from the oracle on %s at H=%d" % (name, H))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--check-reads", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    lines = []

    def emit(rec):
        rec = dict(rec, **info)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    w = synth.WORKLOADS["metagenome"]
    measure("metagenome", synth.generate(w), w.n_snps, (5, 50, 100), args.reps, args.check_reads, emit)
    w = synth.WORKLOADS["ont"]
    measure("ont", synth.generate(w), w.n_snps, (50,), args.reps, args.check_reads, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
