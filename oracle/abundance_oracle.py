"""Read classes and the abundance EM in numpy / plain Python, written from the definition in DESIGN.md §4 K7; the
reference has no counterpart.  Test infrastructure only: the product must not import it.

Read assignment is K5's (oracle/support_oracle.py): for a read (r, c[0..k-1]), c[t] is the allele at site r+t+1,
informative when it is not N (4) or _ (6); d_h = informative t with c[t] != hap[h][r+t+1]; D = min_h d_h;
B = {h : d_h = D}.  Uninformative: no informative site.  Over the limit: max_mismatch >= 0 and D > max_mismatch.
Every other read is assigned and adds 1 to the class keyed by B (ascending).  Classes with a count >= 1 are listed in
lexicographic order of their member lists, as CSR (class_off int64[C+1], members int32[M], count int64[C]).

The EM runs over the classes in that order, in float64, in exactly this operation order (T = the sum of counts):

    pi[h] = 1.0 / H
    for it in 1..max_iter:
        acc[h] = 0.0
        for each class c:  z = sum of pi[h] over members (in member order)
                           acc[h] += float(count[c]) * (pi[h] / z) for each member h
        delta = 0.0
        for h in 0..H-1:   nw = acc[h] / float(T); delta = max(delta, abs(nw - pi[h])); pi[h] = nw
        n_iter = it
        if delta <= tol: break
    loglik = sum over classes of float(count[c]) * log10(z_c), z_c summed as above over the final pi

converged = delta <= tol, where delta is +inf until an iteration has run (max_iter = 0: pi stays uniform and the EM
has not converged).  T = 0: pi all 0, n_iter 0, loglik 0, converged.
"""
from __future__ import annotations

import math

import numpy as np


def _check(haps, rank, off, codes):
    H, N = haps.shape[0], haps.shape[1] - 1
    if H < 1:
        raise ValueError("no haplotype")
    if (haps[:, 1:] > 6).any():
        raise ValueError("haplotype code > 6")
    k = np.diff(off)
    if len(rank) and ((rank < 0).any() or (k < 0).any() or (rank + k > N).any()):
        raise ValueError("a read leaves sites 1..N")
    if len(codes[off[0]:off[-1]]) and codes[off[0]:off[-1]].max() > 6:
        raise ValueError("read code > 6")


def _tie_sets(haps, rank, off, codes, max_mismatch):
    """One chunk of reads -> (tie mask bool [n][H] of the assigned reads, status int64[n]: 0 assigned,
    1 uninformative, 2 over the limit)."""
    H = haps.shape[0]
    k = np.diff(off)
    n = len(k)
    c = codes[off[0]:off[-1]]
    read_of = np.repeat(np.arange(n), k)
    site = rank[read_of] + (np.arange(len(c)) - (off[:-1] - off[0])[read_of]) + 1
    informative = (c != 4) & (c != 6)
    mism = (haps[:, site] != c[None, :]) & informative[None, :]
    d = np.zeros((H, n), np.int64)
    m = np.zeros(n, np.int64)
    nz = np.nonzero(k > 0)[0]
    if len(nz):
        starts = off[nz] - off[0]
        d[:, nz] = np.add.reduceat(mism, starts, axis=1, dtype=np.int32)
        m[nz] = np.add.reduceat(informative, starts, dtype=np.int32)
    D = d.min(axis=0)
    unin = m == 0
    over = ~unin & (max_mismatch >= 0) & (D > max_mismatch)
    status = np.where(unin, 1, np.where(over, 2, 0))
    tied = (d == D[None, :]).T
    return tied[status == 0], status


def _csr(pairs, assigned, uninformative, over_limit):
    """[(member tuple, count)] -> the CSR dict, in lexicographic order of the member lists."""
    pairs = sorted(pairs)
    sizes = [len(b) for b, _ in pairs]
    return {"class_off": np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64),
            "members": np.array([h for b, _ in pairs for h in b], np.int32),
            "count": np.array([n for _, n in pairs], np.int64),
            "assigned": assigned, "uninformative": uninformative, "over_limit": over_limit}


def classes(haps, rank, off, codes, max_mismatch=-1):
    """-> dict(class_off, members, count, assigned, uninformative, over_limit).  Per chunk of about 2^25 / H alleles,
    the tie masks of the assigned reads are packed to bytes and counted by np.unique; the chunks' counts are merged
    the same way, and the member lists are sorted last."""
    haps = np.asarray(haps, dtype=np.uint8)
    rank = np.asarray(rank, dtype=np.int64)
    off = np.asarray(off, dtype=np.int64)
    codes = np.asarray(codes, dtype=np.uint8)
    _check(haps, rank, off, codes)
    H, R = haps.shape[0], len(rank)
    chunk_codes = max(4096, (1 << 25) // H)
    rows, counts, tot = [], [], np.zeros(3, np.int64)
    a = 0
    while a < R:
        b = int(np.searchsorted(off, off[a] + chunk_codes, side="right")) - 1
        b = min(max(b, a + 1), R)
        tied, status = _tie_sets(haps, rank[a:b], off[a:b + 1], codes, max_mismatch)
        tot += np.bincount(status, minlength=3)
        if len(tied):
            u, n = np.unique(np.packbits(tied, axis=1), axis=0, return_counts=True)
            rows.append(u)
            counts.append(n)
        a = b
    pairs = []
    if rows:
        u, inv = np.unique(np.concatenate(rows), axis=0, return_inverse=True)
        n = np.bincount(inv.reshape(-1), weights=np.concatenate(counts), minlength=len(u)).astype(np.int64)
        masks = np.unpackbits(u, axis=1, count=H).astype(bool)
        pairs = [(tuple(int(h) for h in np.nonzero(masks[i])[0]), int(n[i])) for i in range(len(u))]
    return _csr(pairs, int(tot[0]), int(tot[1]), int(tot[2]))


def classes_loop(haps, rank, off, codes, max_mismatch=-1):
    """The same definition as a literal per-read Python loop (small inputs; checks ``classes``)."""
    H = len(haps)
    count, tot = {}, [0, 0, 0]
    for i in range(len(rank)):
        r, c = int(rank[i]), [int(x) for x in codes[off[i]:off[i + 1]]]
        inf = [t for t in range(len(c)) if c[t] not in (4, 6)]
        if not inf:
            tot[1] += 1
            continue
        d = [sum(1 for t in inf if c[t] != int(haps[h][r + t + 1])) for h in range(H)]
        D = min(d)
        if max_mismatch >= 0 and D > max_mismatch:
            tot[2] += 1
            continue
        tot[0] += 1
        B = tuple(h for h in range(H) if d[h] == D)
        count[B] = count.get(B, 0) + 1
    return _csr(list(count.items()), *tot)


def em(n_haps, class_off, members, count, max_iter=10000, tol=1e-12):
    """The EM of the module docstring as a plain loop -> dict(pi list of float, n_iter, converged, loglik)."""
    C = len(count)
    cls = [[int(h) for h in members[class_off[c]:class_off[c + 1]]] for c in range(C)]
    cnt = [int(x) for x in count]
    T = sum(cnt)
    if T == 0:
        return {"pi": [0.0] * n_haps, "n_iter": 0, "converged": True, "loglik": 0.0}
    pi = [1.0 / n_haps] * n_haps
    delta = math.inf
    n_iter = 0
    for it in range(1, max_iter + 1):
        acc = [0.0] * n_haps
        for c in range(C):
            z = 0.0
            for h in cls[c]:
                z += pi[h]
            assert z > 0.0, "a class lost all its mass"
            for h in cls[c]:
                acc[h] += float(cnt[c]) * (pi[h] / z)
        delta = 0.0
        for h in range(n_haps):
            nw = acc[h] / float(T)
            delta = max(delta, abs(nw - pi[h]))
            pi[h] = nw
        n_iter = it
        if delta <= tol:
            break
    loglik = 0.0
    for c in range(C):
        z = 0.0
        for h in cls[c]:
            z += pi[h]
        assert z > 0.0, "a class lost all its mass"
        loglik += float(cnt[c]) * math.log10(z)
    return {"pi": pi, "n_iter": n_iter, "converged": delta <= tol, "loglik": loglik}
