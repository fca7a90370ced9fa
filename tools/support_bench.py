"""Read support (Hansel.assign_reads) on config 3: 10M x 150 bp reads over N = 10k sites, against haplotypes that are
the 5 strains plus random mutants of them, for H in {5, 50, 100}; and the ONT workload at H = 50.

Per H: the assignment kernels' device time (hx_last_kernel_ms(3), best of --reps after a warm-up call), the wall time
of assign_reads from host arrays, reads x haplotypes per second of kernel time, and the host->device copy of the
packed reads from pinned memory (CUDA events) for comparison.  The oracle (oracle/support_oracle.py) checks the
result on a 1M-read subsample.  Card name and power limit are read in the same run.  One JSON line per measurement;
--out also writes them to a file.

    python tools/support_bench.py [--reps 10] [--out results/support_bench.jsonl]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from gretel_b200 import synth  # noqa: E402
from gretel_b200.hansel import REF_SYMBOLS, REF_UNSYMBOLS, Hansel  # noqa: E402
from oracle import support_oracle as so  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split(",")[:2]]
    return {"gpu": name, "power_limit": power}


def haplotypes(strains, H, seed=11, rate=0.01):
    rng = np.random.default_rng(seed)
    base = np.concatenate([np.full((len(strains), 1), 6, np.uint8), strains], axis=1)
    rows = [base[i % len(base)].copy() for i in range(H)]
    for i in range(len(base), H):
        hit = np.nonzero(rng.random(base.shape[1] - 1) < rate)[0] + 1
        rows[i][hit] = (rows[i][hit] + rng.integers(1, 4, size=len(hit))) % 4
    return np.stack(rows)


def copy_ms(d, reps):
    """Host->device copy of the packed reads (rank, off, codes) from pinned memory, best of reps."""
    import torch
    src = [torch.from_numpy(np.ascontiguousarray(d[k])).pin_memory() for k in ("rank", "off", "codes")]
    dst = [torch.empty_like(s, device="cuda") for s in src]
    best = float("inf")
    for _ in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for s, t in zip(src, dst):
            t.copy_(s, non_blocking=True)
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best, sum(s.numel() * s.element_size() for s in src)


def measure(name, d, N, Hs, reps, check_reads, emit):
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=1, device=0)
    rank, off, codes = d["rank"], d["off"], d["codes"]
    R = len(rank)
    cms, nbytes = copy_ms(d, reps)
    for H in Hs:
        haps = haplotypes(d["strains"], H)
        res = h.assign_reads(haps, rank, off, codes)                 # warm-up
        kern, wall = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            h.assign_reads(haps, rank, off, codes)
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(h.kernel_ms("assign"))
        # the oracle on a subsample of reads (the first check_reads)
        n = min(R, check_reads)
        sub = h.assign_reads(haps, rank[:n], off[:n + 1], codes, per_read=True)
        exp = so.assign(haps, rank[:n], off[:n + 1], codes)
        equal = all(np.array_equal(np.asarray(getattr(sub, f)), np.asarray(exp[f])) for f in
                    ("unique", "shared", "share_q32", "assigned", "uninformative", "over_limit", "best_mm", "n_best",
                     "first_best"))
        emit({"workload": name, "reads": R, "codes": int(off[-1] - off[0]), "H": H, "kernel_ms": min(kern),
              "kernel_ms_median": float(np.median(kern)), "wall_ms": min(wall), "wall_ms_median": float(np.median(wall)),
              "reads_x_haps_per_s": R * H / (min(kern) * 1e-3), "h2d_copy_ms_pinned": cms, "h2d_bytes": nbytes,
              "assigned": res.assigned, "uninformative": res.uninformative, "oracle_reads": n, "oracle_equal": equal})
        if not equal:
            raise SystemExit("read support differs from the oracle on %s at H=%d" % (name, H))


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
