"""Recovery entry points with the reference's names, arguments and return values.

Mirrors gretel/gretel.py:13 (reweight_hansel_from_path) and :102 (generate_path); the
whole per-site walk and the O(N*W) reweight run on the GPU with no host round trip
per site.  ``recover`` is the driver loop of gretel/cmd.py:148-179.
"""
from __future__ import annotations

import sys

import numpy as np


def reweight_hansel_from_path(hansel, path, ratio):
    """gretel/gretel.py:13-98 -> sum of removed observations (float)."""
    size = hansel.reweight_path_codes(hansel.encode_path(path), ratio)
    sys.stderr.write("[RWGT] Ratio %.3f, Removed %.1f\n" % (ratio, size))
    return size


def generate_path(n_snps, hansel, original_hansel, debug_hpos=None):
    """gretel/gretel.py:102-189 -> (path, {"hp_original","hp_current"}, min_marginal)
    or (None, None, None) when a hole is found (gretel.py:176-180)."""
    if n_snps != hansel.n_snps:
        raise ValueError("n_snps does not match the Hansel matrix")
    sys.stderr.write("[NOTE] *Establishing next path\n")
    res = hansel.generate_path_codes(original_hansel)
    if res[0] is None:
        snp = res[1]
        sys.stderr.write('''[NOTE] Unable to select next branch from SNP %d to %d
       By design, Gretel will attempt to recover haplotypes until a hole in the graph has been found.
       Recovery will intentionally terminate now.\n''' % (snp - 1, snp))
        return None, None, None
    codes, hp_cur, hp_orig, min_marg = res
    if debug_hpos:
        path = hansel.decode_path(codes)
        for snp in debug_hpos:
            if 1 <= snp <= n_snps:
                print(hansel.get_edge_weights_at(snp, path))
    return hansel.decode_path(codes), {"hp_original": hp_orig, "hp_current": hp_cur}, min_marg


def recover(hansel, n_snps, max_paths=100, min_remove=0.01, original_hansel=None, resident=True):
    """gretel/cmd.py:79,148-179: copy, up to ``max_paths`` x (generate, clamp ratio,
    reweight), PATHS bookkeeping.  ``resident=True`` keeps the loop on the device
    (hx_recover); ``False`` calls generate_path / reweight_hansel_from_path per haplotype
    exactly like cmd.py does.  Returns (iterations, PATHS)."""
    original = original_hansel if original_hansel is not None else hansel.copy()
    iters = []
    if resident:
        codes, stats = hansel.recover_codes(original, max_paths, min_remove)
        for c, s in zip(codes, stats):
            iters.append({"hansel_path": hansel.decode_path(c), "hp_current": float(s[0]),
                          "hp_original": float(s[1]), "min_marginal": float(s[2]), "ratio": float(s[3]),
                          "removed": float(s[4])})
    else:
        for _ in range(max_paths):
            path, prob, init_min = generate_path(n_snps, hansel, original)
            if path is None:
                break
            ratio = init_min
            if ratio < min_remove:
                sys.stderr.write("[RWGT] Ratio %.10f too small, adjusting to %.3f\n" % (ratio, min_remove))
                ratio = min_remove
            mag = reweight_hansel_from_path(hansel, path, ratio)
            iters.append({"hansel_path": path, "hp_current": prob["hp_current"],
                          "hp_original": prob["hp_original"], "min_marginal": init_min, "ratio": ratio,
                          "removed": mag})
    PATHS = {}
    for i, it in enumerate(iters):
        key = "".join(str(x) for x in it["hansel_path"])
        it["path"] = key
        if key not in PATHS:
            PATHS[key] = {"hp_current": [], "hp_original": [], "i": [], "i_0": i, "n": 0, "magnitude": 0,
                          "hansel_path": it["hansel_path"]}
        PATHS[key]["n"] += 1
        PATHS[key]["i"].append(i)
        PATHS[key]["magnitude"] += it["removed"]
        PATHS[key]["hp_current"].append(it["hp_current"])
        PATHS[key]["hp_original"].append(it["hp_original"])
    return iters, PATHS


def gap_check(hansel, n_snps):
    """gretel/cmd.py:85-92: sites whose pairwise evidence total is zero."""
    return [i for i in range(0, n_snps + 1) if hansel.get_counts_at(i).get("total", 0) == 0]


def read_support(hansel, PATHS, rank, off, codes, max_mismatch=-1):
    """Reads carried by each recovered haplotype: the packed reads are assigned to the distinct paths of ``PATHS``
    (Hansel.assign_reads) in ``i_0`` order, the order of out.fasta.  Returns (records, totals): one dict per path
    with i_0, unique, shared, share and share_q32, and a dict with reads, assigned, uninformative, over_limit and
    max_mismatch.  With no path no read is assigned: reads without an informative site are uninformative, the
    others over the limit."""
    keys = sorted(PATHS, key=lambda x: PATHS[x]["i_0"])
    totals = {"reads": len(rank), "max_mismatch": int(max_mismatch)}
    if not keys:
        off = np.asarray(off, dtype=np.int64)
        informative = np.concatenate([[0], np.cumsum(np.isin(codes[off[0]:off[-1]], (4, 6), invert=True))])
        n_unin = int((np.diff(informative[off - off[0]]) == 0).sum())
        totals.update(assigned=0, uninformative=n_unin, over_limit=len(rank) - n_unin)
        return [], totals
    paths = np.stack([hansel.encode_path(PATHS[k]["hansel_path"]) for k in keys])
    res = hansel.assign_reads(paths, rank, off, codes, max_mismatch=max_mismatch)
    totals.update(assigned=res.assigned, uninformative=res.uninformative, over_limit=res.over_limit)
    records = [{"i_0": PATHS[k]["i_0"], "unique": int(res.unique[j]), "shared": int(res.shared[j]),
                "share": float(res.share[j]), "share_q32": int(res.share_q32[j])} for j, k in enumerate(keys)]
    return records, totals


def abundance(hansel, PATHS, rank, off, codes, max_mismatch=-1, max_iter=10000, tol=1e-12, n_boot=0, seed=0):
    """How abundant each recovered haplotype is: the packed reads are grouped into compatibility classes over the
    distinct paths of ``PATHS`` (Hansel.read_classes) and each path's share of the assigned reads is estimated by EM
    over the classes (hansel.em_abundance).  Unlike read_support's equal split, a read tied between paths goes to
    them in proportion to their estimated abundance.  Returns (records, totals): one dict per path in ``i_0`` order
    with i_0, unique, shared, em_reads (= em_fraction * assigned) and em_fraction, and a dict with reads, assigned,
    uninformative, over_limit, max_mismatch, classes, iterations, converged and loglik.  With no path no read is
    assigned, as in read_support.  With ``n_boot`` > 0 the EM is also run on ``n_boot`` bootstrap resamples of the
    assigned reads on the GPU (Hansel.em_bootstrap with ``seed``): each record gains boot_mean, boot_sd (ddof = 1; 0
    for one replicate), boot_lo and boot_hi (the 2.5 % and 97.5 % quantiles) of its fraction over the replicates,
    and the totals gain replicates, seed and boot_converged (the replicates whose EM converged).  The point estimate
    stays em_abundance's."""
    from .hansel import em_abundance
    keys = sorted(PATHS, key=lambda x: PATHS[x]["i_0"])
    if not keys:
        _, totals = read_support(hansel, PATHS, rank, off, codes, max_mismatch=max_mismatch)
        totals.update(classes=0, iterations=0, converged=True, loglik=0.0)
        if n_boot > 0:
            totals.update(replicates=int(n_boot), seed=int(seed), boot_converged=int(n_boot))
        return [], totals
    paths = np.stack([hansel.encode_path(PATHS[k]["hansel_path"]) for k in keys])
    cls = hansel.read_classes(paths, rank, off, codes, max_mismatch=max_mismatch)
    em = em_abundance(len(keys), cls, max_iter=max_iter, tol=tol)
    size = np.diff(cls.class_off)
    of_class = np.repeat(np.arange(len(cls)), size)
    unique = np.bincount(cls.members[size[of_class] == 1], weights=cls.count[of_class][size[of_class] == 1],
                         minlength=len(keys)).astype(np.int64)
    shared = np.bincount(cls.members[size[of_class] >= 2], weights=cls.count[of_class][size[of_class] >= 2],
                         minlength=len(keys)).astype(np.int64)
    totals = {"reads": len(rank), "assigned": cls.assigned, "uninformative": cls.uninformative,
              "over_limit": cls.over_limit, "max_mismatch": int(max_mismatch), "classes": len(cls),
              "iterations": em.n_iter, "converged": em.converged, "loglik": em.loglik}
    records = [{"i_0": PATHS[k]["i_0"], "unique": int(unique[j]), "shared": int(shared[j]),
                "em_reads": float(em.pi[j] * cls.assigned), "em_fraction": float(em.pi[j])}
               for j, k in enumerate(keys)]
    if n_boot > 0:
        boot = hansel.em_bootstrap(len(keys), cls, n_boot, seed=seed, max_iter=max_iter, tol=tol)
        for j, r in enumerate(records):
            r.update(boot_summary(boot.pi[1:, j]))
        totals.update(replicates=int(n_boot), seed=int(seed), boot_converged=int(boot.converged[1:].sum()))
    return records, totals


def boot_summary(x):
    """boot_mean, boot_sd (ddof = 1, 0.0 for one value), boot_lo and boot_hi (the 2.5 % and 97.5 % quantiles) of the
    replicate fractions ``x``."""
    return {"boot_mean": float(np.mean(x)), "boot_sd": float(np.std(x, ddof=1)) if len(x) > 1 else 0.0,
            "boot_lo": float(np.quantile(x, 0.025)), "boot_hi": float(np.quantile(x, 0.975))}


def score_paths(hansel, PATHS, weights=False):
    """Score the distinct recovered paths of ``PATHS`` in ``i_0`` order (the order of out.fasta) against ``hansel``
    (Hansel.score_paths).  Score against the matrix recovery started from (``original_hansel``): recovery reweights
    the matrix it walks.  Returns (i_0 list, paths uint8 [H][N+1], PathScores); ([], None, None) without a path."""
    keys = sorted(PATHS, key=lambda x: PATHS[x]["i_0"])
    if not keys:
        return [], None, None
    paths = np.stack([hansel.encode_path(PATHS[k]["hansel_path"]) for k in keys])
    return [PATHS[k]["i_0"] for k in keys], paths, hansel.score_paths(paths, weights=weights)


def sequence_path(seq, vcf_h, delchar=""):
    """A known sequence (same coordinates as --master) as a path: '_', then per site j the character at 1-based
    position snp_rev[j] - A, C, G or T (either case) as itself, ``delchar`` (if not empty) as '-', anything else,
    or a position past the end of the sequence, as N.  -> uint8 [N+1]."""
    code = {"A": 0, "C": 1, "G": 2, "T": 3}
    out = np.full(vcf_h["N"] + 1, 4, dtype=np.uint8)
    out[0] = 6
    for j in range(vcf_h["N"]):
        pos = vcf_h["snp_rev"][j]
        ch = seq[pos - 1] if 1 <= pos <= len(seq) else ""
        if delchar and ch == delchar:
            out[j + 1] = 5
        else:
            out[j + 1] = code.get(ch.upper(), 4)
    return out


def score_sequences(hansel, vcf_h, fasta_records, delchar="", weights=False):
    """Score known sequences ((name, sequence) pairs, e.g. reference strains from a panel) as paths (sequence_path)
    against ``hansel``.  Returns (names, paths uint8 [H][N+1], PathScores); ([], None, None) without a record."""
    if not fasta_records:
        return [], None, None
    paths = np.stack([sequence_path(seq, vcf_h, delchar) for _, seq in fasta_records])
    return [name for name, _ in fasta_records], paths, hansel.score_paths(paths, weights=weights)
