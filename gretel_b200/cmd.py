"""Command-line driver with the reference's flags and outputs (gretel/cmd.py:11-240), on the B200 path.

    python -m gretel_b200 <bam> <vcf.gz> <contig> [-s START] [-e END] [-p PATHS] [-o OUT] ...

Everything that computes (ingestion, gap check counts, recovery, reweighting) runs in the CUDA
library; this file is host-side bookkeeping and output formatting only: PATHS de-duplication
(cmd.py:164-179), out.fasta / snp.fasta (cmd.py:181-221) and gretel.crumbs (cmd.py:223-240,
docs/protocol.rst:48-77), and with --support the reads carried by each haplotype (gretel.support, no reference
counterpart); with --site-weights / --score the branch weights of every recovered haplotype and of known sequences,
site by site (gretel.sites, gretel.scores, no reference counterpart).
"""
from __future__ import annotations

import argparse
import sys

from . import gretel, util

__version__ = "0.0.94+b200"


def read_first_fasta_record(path):
    """First sequence of a FASTA file (the reference uses pysam.FastaFile, util.py:337-351)."""
    seq = []
    seen = False
    with open(path) as fh:
        for line in fh:
            if line.startswith(">"):
                if seen:
                    break
                seen = True
                continue
            if seen:
                seq.append(line.strip())
    return "".join(seq)


def read_fasta_records(path):
    """Every record of a FASTA file as (name, sequence); the name is the header up to the first whitespace."""
    records, name, seq = [], None, []
    with open(path) as fh:
        for line in fh:
            if line.startswith(">"):
                if name is not None:
                    records.append((name, "".join(seq)))
                name, seq = (line[1:].split() or [""])[0], []
            elif name is not None:
                seq.append(line.strip())
    if name is not None:
        records.append((name, "".join(seq)))
    return records


def build_parser():
    p = argparse.ArgumentParser(prog="gretel", description="Gretel: A metagenomic haplotyper (B200 hot path).")
    p.add_argument("bam")
    p.add_argument("vcf")
    p.add_argument("contig")
    p.add_argument("-s", "--start", type=int, default=1)
    p.add_argument("-e", "--end", type=int, default=-1)
    p.add_argument("-p", "--paths", type=int, default=100)
    p.add_argument("--master", default=None)
    p.add_argument("--gapchar", default="N")
    p.add_argument("--delchar", default="")
    p.add_argument("--quiet", default=False, action="store_true")
    p.add_argument("-o", "--out", default=".")
    p.add_argument("-@", "--threads", type=int, default=1)
    p.add_argument("--dumpmatrix", type=str, default=None)
    p.add_argument("--dumpsnps", type=str, default=None)
    p.add_argument("--pepper", action="store_true")
    p.add_argument("--device", type=int, default=None)
    p.add_argument("--support", action="store_true",
                   help="write gretel.support: the reads each recovered haplotype carries")
    p.add_argument("--max-mismatch", type=int, default=-1,
                   help="--support: a read whose best haplotype has more mismatches is not assigned (-1: no limit)")
    p.add_argument("--site-weights", action="store_true",
                   help="write gretel.sites: per recovered haplotype and site the branch weights of its allele, of "
                        "the best candidate and of the runner-up; and gretel.scores: per haplotype its log "
                        "likelihood, unsupported sites and sites where another allele is preferred")
    p.add_argument("--score", default=None, metavar="FASTA",
                   help="also score every record of FASTA (same coordinates as --master) against the evidence, in "
                        "gretel.scores (and gretel.sites with --site-weights)")
    p.add_argument("--version", action="version", version="%(prog)s " + __version__)
    return p


def snp_table(hansel, vcf_h, out=sys.stdout):
    """cmd.py:123-145."""
    out.write("i\tpos\tgap\tA\tC\tG\tT\tN\t-\t_\ttot\n")
    last_rev = 0
    for i in range(0, vcf_h["N"] + 1):
        m = {str(k): v for k, v in hansel.get_counts_at(i).items()}
        snp_rev = vcf_h["snp_rev"][i - 1] if i > 0 else 0
        out.write("%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\n" % (
            i, snp_rev, snp_rev - last_rev, m.get("A", 0), m.get("C", 0), m.get("G", 0), m.get("T", 0),
            m.get("N", 0), m.get("-", 0), m.get("_", 0), m.get("total", 0)))
        last_rev = snp_rev


def write_outputs(dirn, PATHS, hansel, vcf_h, start, end, master=None, gapchar="N", delchar=""):
    """cmd.py:181-240: out.fasta, snp.fasta, gretel.crumbs."""
    dirn = dirn.rstrip("/") + "/"
    master_seq = read_first_fasta_record(master) if master else [' '] * end
    with open(dirn + "out.fasta", "w") as fasta, open(dirn + "snp.fasta", "w") as hfasta:
        for key in sorted(PATHS, key=lambda x: PATHS[x]["i_0"]):
            p = PATHS[key]
            path, i = p["hansel_path"], p["i_0"]
            seq = list(master_seq[:])
            for j, mallele in enumerate(path[1:]):
                pos = vcf_h["snp_rev"][j]
                seq[pos - 1] = delchar if mallele == hansel.symbols_d["-"] else mallele
            to_write = "".join(str(x) for x in seq[start - 1:end])
            if not master:
                to_write = to_write.replace(' ', gapchar)
            fasta.write(">%d__%.2f\n%s\n" % (i, p["hp_current"][0], to_write))
            hfasta.write(">%d__%.2f\n%s\n" % (i, p["hp_current"][0], "".join(str(x) for x in path[1:])))
    with open(dirn + "gretel.crumbs", "w") as crumbs:
        crumbs.write("# %d\t%d\t%d\t%.2f\n" % (vcf_h["N"], hansel.n_crumbs, hansel.n_slices, hansel.L))
        for key in sorted(PATHS, key=lambda x: PATHS[x]["hp_current"][0], reverse=True):
            p = PATHS[key]
            crumbs.write("%d\t%d\t%s\t%s\t%.2f\n" % (
                p["i_0"], p["n"], ",".join("%.2f" % x for x in p["hp_current"]),
                ",".join("%.2f" % x for x in p["hp_original"]), p["magnitude"]))


def write_support(dirn, records, totals):
    """gretel.support: '# reads, assigned, uninformative, over_limit, max_mismatch', then per distinct haplotype in
    i_0 order: i_0, unique reads, shared reads, share of the reads, share / assigned."""
    with open(dirn.rstrip("/") + "/gretel.support", "w") as fh:
        fh.write("# %d\t%d\t%d\t%d\t%d\n" % (totals["reads"], totals["assigned"], totals["uninformative"],
                                             totals["over_limit"], totals["max_mismatch"]))
        for r in records:
            fh.write("%d\t%d\t%d\t%.2f\t%.4f\n" % (r["i_0"], r["unique"], r["shared"], r["share"],
                                                 r["share"] / totals["assigned"] if totals["assigned"] else 0.0))


def write_scores(dirn, hansel, vcf_h, scored, site_weights):
    """gretel.scores: per scored path (recovered ones by i_0, then FASTA records by name) loglik, unsupported sites
    and sites whose best candidate is not the path's allele.  With site_weights, gretel.sites: per path and site
    the site, its position, the path's allele, its weight, the best candidate (. if none), its weight and the largest
    weight of the candidates other than the path's allele.  `scored`: (keys, paths uint8 [H][N+1], PathScores)
    blocks as gretel.score_paths / score_sequences return them.  Weights are written in full precision (repr)."""
    dirn = dirn.rstrip("/") + "/"
    with open(dirn + "gretel.scores", "w") as fh:
        fh.write("#id\tloglik\tn_unsupported\tn_disagree\n")
        for keys, _, sc in scored:
            for j, k in enumerate(keys):
                fh.write("%s\t%r\t%d\t%d\n" % (k, float(sc.loglik[j]), sc.n_unsupported[j], sc.n_disagree[j]))
    if not site_weights:
        return
    sym = hansel.symbols
    with open(dirn + "gretel.sites", "w") as fh:
        fh.write("#id\tsite\tpos\tallele\tw_hap\tbest\tw_best\tw_second\n")
        for keys, paths, sc in scored:
            for j, k in enumerate(keys):
                for s in range(1, vcf_h["N"] + 1):
                    b = int(sc.best[j, s - 1])
                    none = b == sc.NO_CANDIDATE
                    fh.write("%s\t%d\t%d\t%s\t%r\t%s\t%r\t%r\n" % (
                        k, s, vcf_h["snp_rev"][s - 1], sym[paths[j][s]], float(sc.w_hap[j, s - 1]),
                        "." if none else sym[b], 0.0 if none else float(sc.weights[j, s - 1, b]),
                        float(sc.w_second[j, s - 1])))


def main(argv=None):
    args = build_parser().parse_args(argv)
    if args.end == -1:
        args.end = util.get_ref_len_from_bam(args.bam, args.contig)
        sys.stderr.write("[NOTE] Setting end_pos to %d" % args.end)
    vcf_h = util.process_vcf(args.vcf, args.contig, args.start, args.end)
    if args.dumpsnps:
        with open(args.dumpsnps, "w") as fh:
            for k in sorted(vcf_h["snp_fwd"].keys()):
                fh.write("%d\t%d\t%d\n" % (vcf_h["snp_fwd"][k] + 1, k, k - args.start + 1))
    reads = {} if args.support else None
    hansel = util.load_from_bam(args.bam, args.contig, args.start, args.end, vcf_h, n_threads=args.threads,
                                stepper="all" if args.pepper else "samtools", device=args.device, reads=reads)
    if args.dumpmatrix:
        hansel.save_hansel_dump(args.dumpmatrix)
    gaps = gretel.gap_check(hansel, vcf_h["N"])
    if gaps:
        i = gaps[0]
        sys.stderr.write("[FAIL] Unable to recover pairwise evidence concerning SNP #%d at position %d\n" % (
            i, vcf_h["snp_rev"][i - 1] if i > 0 else 0))
        return 1
    if not args.quiet:
        snp_table(hansel, vcf_h)
    original = hansel.copy()                      # what recovery starts from: paths are scored against it
    _, PATHS = gretel.recover(hansel, vcf_h["N"], max_paths=args.paths, min_remove=0.01, original_hansel=original)
    write_outputs(args.out, PATHS, hansel, vcf_h, args.start, args.end, master=args.master,
                  gapchar=args.gapchar, delchar=args.delchar)
    if args.support:
        records, totals = gretel.read_support(hansel, PATHS, reads["rank"], reads["off"], reads["codes"],
                                              max_mismatch=args.max_mismatch)
        write_support(args.out, records, totals)
    if args.site_weights or args.score:
        scored = [gretel.score_paths(original, PATHS, weights=args.site_weights)]
        if args.score:
            scored.append(gretel.score_sequences(original, vcf_h, read_fasta_records(args.score),
                                                 delchar=args.delchar, weights=args.site_weights))
        write_scores(args.out, original, vcf_h, [s for s in scored if s[0]], args.site_weights)
    return 0


if __name__ == "__main__":
    sys.exit(main())
