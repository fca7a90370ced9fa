"""Path scores (Hansel.score_paths) against the recovery of the same haplotypes: config 3 (10M x 150 bp reads, N = 10k,
L = 15) at H = 5, 50 and 100, and the ONT workload (L ~ 290) at H = 50.

The haplotypes are the first H that hx_recover finds on the matrix; recovery time is hx_last_kernel_ms(1) of that
hx_recover call (device time of the whole resident loop).  Scoring is timed with hx_last_kernel_ms(4) (the scoring
kernels, copies excluded), best of --reps after a warm-up call, for the default term path and for each path forced
with HX_SCORE_TABLES; the wall time of score_paths from host arrays is reported beside it.  Both paths must give the
same bytes, and the first haplotype must score n_disagree = 0 on the matrix it was walked on.  Card name and power
limit are read in the same run.  One JSON line per measurement; --out also writes them to a file.

    python tools/score_bench.py [--reps 10] [--out results/score_bench.jsonl]
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

from gretel_b200 import synth, util  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = [x.strip() for x in q.stdout.strip().split(",")[:2]]
    return {"gpu": name, "power_limit": power}


def timed_scores(h, paths, reps, tables):
    if tables is None:
        os.environ.pop("HX_SCORE_TABLES", None)
    else:
        os.environ["HX_SCORE_TABLES"] = str(int(tables))
    try:
        res = h.score_paths(paths)                                    # warm-up
        kern, wall = [], []
        for _ in range(reps):
            t0 = time.perf_counter()
            res = h.score_paths(paths)
            wall.append((time.perf_counter() - t0) * 1e3)
            kern.append(h.kernel_ms("score"))
    finally:
        os.environ.pop("HX_SCORE_TABLES", None)
    return res, min(kern), float(np.median(kern)), min(wall)


def measure(name, d, N, Hs, reps, emit):
    h = util.load_from_packed(d["rank"], d["off"], d["codes"], N, band_w=d["max_k"] - 1)
    L = h.L
    recov = {}
    for H in Hs:
        work = h.copy()
        paths, _ = work.recover_codes(h, H, 0.01)
        recov[H] = (paths, work.kernel_ms("walk"))
        work.close()
    for H in Hs:
        paths, rec_ms = recov[H]
        n = len(paths)
        out = {}
        for mode, tables in (("default", None), ("tables", True), ("band", False)):
            if mode == "tables" and L > 32 and n > 5:
                continue                                            # ONT tables: (N+2) x L x 448 B; not the default
            out[mode] = timed_scores(h, paths, reps, tables)
        ref = out["default"][0]
        equal = all(np.array_equal(getattr(r[0], f), getattr(ref, f)) for r in out.values()
                    for f in ("w_hap", "w_second", "best", "loglik", "n_unsupported", "n_disagree"))
        rec = {"workload": name, "N": N, "L": L, "W": h.band_w, "H": n, "recovery_ms": rec_ms,
               "paths_equal": equal, "first_n_disagree": int(ref.n_disagree[0])}
        for mode, (_, kbest, kmed, wall) in out.items():
            rec.update({"%s_kernel_ms" % mode: kbest, "%s_kernel_ms_median" % mode: kmed, "%s_wall_ms" % mode: wall,
                        "%s_ns_per_hap_site" % mode: kbest * 1e6 / (n * N)})
        rec["score_over_recovery"] = out["default"][1] / rec_ms if rec_ms > 0 else None
        emit(rec)
        if not equal or ref.n_disagree[0] != 0:
            raise SystemExit("score paths differ, or the first haplotype disagrees with its walk (%s, H=%d)" % (name, n))
    h.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    info = card()
    lines = []

    def emit(rec):
        rec = dict(rec, **info)
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)

    w = synth.WORKLOADS["metagenome"]
    measure("metagenome", synth.generate(w), w.n_snps, (5, 50, 100), args.reps, emit)
    w = synth.WORKLOADS["ont"]
    measure("ont", synth.generate(w), w.n_snps, (50,), args.reps, emit)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
