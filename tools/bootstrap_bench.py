"""Bootstrap of the abundance EM (Hansel.em_bootstrap) on the classes of tools/abundance_bench.py: config 3 (10M x 150 bp
reads over N = 10k sites) against the 5 strains plus random mutants of them for H in {5, 50, 100}, and the ONT
workload at H = 50; each at B in {0, 100, 1000} replicates.

Per row: the resampling and EM kernels' device time (hx_last_kernel_ms(6), (7); best of --reps after a warm-up call),
the wall time of em_bootstrap, the host em_abundance on the same classes, the largest and median iteration counts
over the replicates and the replicates that converged.  Checked in the same run: row 0 equals the host EM bit for
bit, the counts of replicates 1 and B equal the numpy resampler (oracle/bootstrap_oracle.py), and the EMs of up to 20
replicates equal the host EM on the classes they keep.  Card name and power limit are read in the same run.  One JSON
line per measurement; --out also writes them to a file.

    python tools/bootstrap_bench.py [--reps 5] [--out results/bootstrap_bench.jsonl]
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
from oracle import bootstrap_oracle as bo  # noqa: E402
from support_bench import card, haplotypes  # noqa: E402


def same(a, pi, it, conv, ll):
    return (a.pi.tobytes() == np.asarray(pi).tobytes() and a.n_iter == int(it) and a.converged == bool(conv)
            and np.float64(a.loglik).tobytes() == np.float64(ll).tobytes())


def measure(name, d, N, Hs, Bs, reps, emit):
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=1, device=0)
    rank, off, codes = d["rank"], d["off"], d["codes"]
    for H in Hs:
        cls = h.read_classes(haplotypes(d["strains"], H), rank, off, codes)
        host_ms = []
        for _ in range(3):
            t0 = time.perf_counter()
            em = em_abundance(H, cls)
            host_ms.append((time.perf_counter() - t0) * 1e3)
        for B in Bs:
            h.em_bootstrap(H, cls, B, seed=1)                             # warm-up
            res, em_k, wall = [], [], []
            for _ in range(reps):
                t0 = time.perf_counter()
                bs = h.em_bootstrap(H, cls, B, seed=1)
                wall.append((time.perf_counter() - t0) * 1e3)
                res.append(h.kernel_ms("resample"))
                em_k.append(h.kernel_ms("bootstrap_em"))
            bs = h.em_bootstrap(H, cls, B, seed=1, counts=True)
            ok0 = same(em, bs.pi[0], bs.n_iter[0], bs.converged[0], bs.loglik[0])
            ok_counts = all(np.array_equal(bs.count[b], bo.resample(cls.count, 1, b)) for b in sorted({1, B}) if B)
            ok_reps = True
            for b in range(1, min(B, 20) + 1):
                fo, fm, fc = bo.filtered(cls.class_off, cls.members, bs.count[b])
                ok_reps &= same(em_abundance(H, (fo, fm, fc)), bs.pi[b], bs.n_iter[b], bs.converged[b], bs.loglik[b])
            emit({"workload": name, "H": H, "B": B, "classes": len(cls), "members": len(cls.members),
                  "assigned": cls.assigned, "resample_kernel_ms": min(res), "em_kernel_ms": min(em_k),
                  "em_kernel_ms_median": float(np.median(em_k)), "wall_ms": min(wall),
                  "wall_ms_median": float(np.median(wall)), "host_em_ms": min(host_ms), "host_em_iterations": em.n_iter,
                  "max_iterations": int(bs.n_iter.max()), "median_iterations": float(np.median(bs.n_iter)),
                  "converged_replicates": int(bs.converged[1:].sum()), "row0_equals_host": ok0,
                  "counts_equal_oracle": ok_counts, "replicates_equal_host": ok_reps})
            if not (ok0 and ok_counts and ok_reps):
                raise SystemExit("bootstrap differs from the host EM or the resampler on %s at H=%d B=%d" % (name, H, B))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--boots", default="0,100,1000")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    lines = []
    Bs = [int(x) for x in args.boots.split(",")]

    def emit(rec):
        rec = dict(rec, **info)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    w = synth.WORKLOADS["metagenome"]
    measure("metagenome", synth.generate(w), w.n_snps, (5, 50, 100), Bs, args.reps, emit)
    w = synth.WORKLOADS["ont"]
    measure("ont", synth.generate(w), w.n_snps, (50,), Bs, args.reps, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
