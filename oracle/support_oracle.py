"""Read support for recovered haplotypes in numpy, written from the definition in DESIGN.md ("Read support");
the reference has no counterpart.  Test infrastructure only: the product must not import it.

For a read (r, c[0..k-1]), c[t] is the allele at site r+t+1.  Site t is informative when c[t] is not N (4) or
_ (6); m = the informative sites.  d_h = informative t with c[t] != hap[h][r+t+1] (plain code equality).
D = min_h d_h, B = {h : d_h = D}, first = min B.  Uninformative: m = 0.  Over the limit: m > 0, max_mismatch >= 0
and D > max_mismatch.  Otherwise assigned.  Over assigned reads: unique[h] counts B = {h}, shared[h] counts
h in B with |B| >= 2, share_q32[h] sums floor(2^32 / |B|) over h in B.
"""
from __future__ import annotations

import numpy as np

Q32 = 1 << 32


def assign(haps, rank, off, codes, max_mismatch=-1):
    """-> dict(unique int64[H], shared int64[H], share_q32 uint64[H], assigned, uninformative, over_limit,
    best_mm, n_best, first_best int32[R]).  Reads go in chunks of about 2^25 / H alleles (bounded temporaries)."""
    haps = np.asarray(haps, dtype=np.uint8)
    rank = np.asarray(rank, dtype=np.int64)
    off = np.asarray(off, dtype=np.int64)
    codes = np.asarray(codes, dtype=np.uint8)
    H, N = haps.shape[0], haps.shape[1] - 1
    R = len(rank)
    chunk_codes = max(4096, (1 << 25) // max(H, 1))
    if H < 1:
        raise ValueError("no haplotype")
    if (haps[:, 1:] > 6).any():
        raise ValueError("haplotype code > 6")
    k = np.diff(off)
    if R and ((rank < 0).any() or (k < 0).any() or (rank + k > N).any()):
        raise ValueError("a read leaves sites 1..N")
    if len(codes[off[0]:off[-1]]) and codes[off[0]:off[-1]].max() > 6:
        raise ValueError("read code > 6")
    out = {"unique": np.zeros(H, np.int64), "shared": np.zeros(H, np.int64), "share_q32": np.zeros(H, np.uint64),
           "best_mm": np.full(R, -1, np.int32), "n_best": np.zeros(R, np.int32), "first_best": np.full(R, -1, np.int32)}
    status = np.zeros(R, np.int64)                               # 0 assigned, 1 uninformative, 2 over the limit
    a = 0
    while a < R:
        b = int(np.searchsorted(off, off[a] + chunk_codes, side="right")) - 1
        b = min(max(b, a + 1), R)
        _chunk(haps, rank[a:b], off[a:b + 1], codes, max_mismatch, out, status[a:b], a)
        a = b
    out["assigned"] = int((status == 0).sum())
    out["uninformative"] = int((status == 1).sum())
    out["over_limit"] = int((status == 2).sum())
    return out


def _chunk(haps, rank, off, codes, max_mismatch, out, status, a):
    H = haps.shape[0]
    k = np.diff(off)
    n = len(k)
    c = codes[off[0]:off[-1]]
    read_of = np.repeat(np.arange(n), k)
    site = rank[read_of] + (np.arange(len(c)) - (off[:-1] - off[0])[read_of]) + 1
    informative = (c != 4) & (c != 6)
    mism = (haps[:, site] != c[None, :]) & informative[None, :]              # [H][codes of the chunk]
    d = np.zeros((H, n), np.int64)
    m = np.zeros(n, np.int64)
    nz = np.nonzero(k > 0)[0]                  # reduceat needs non-empty segments: the reads without codes stay 0
    if len(nz):
        starts = off[nz] - off[0]
        d[:, nz] = np.add.reduceat(mism, starts, axis=1, dtype=np.int32)
        m[nz] = np.add.reduceat(informative, starts, dtype=np.int32)
    D = d.min(axis=0)
    tied = d == D[None, :]
    nb = tied.sum(axis=0)
    first = tied.argmax(axis=0)
    unin = m == 0
    over = ~unin & (max_mismatch >= 0) & (D > max_mismatch)
    asg = ~unin & ~over
    status[unin] = 1
    status[over] = 2
    sl = slice(a, a + n)
    out["best_mm"][sl] = np.where(unin, -1, D)
    out["n_best"][sl] = np.where(unin, 0, nb)
    out["first_best"][sl] = np.where(asg, first, -1)
    t = tied & asg[None, :]
    out["unique"] += (t & (nb == 1)[None, :]).sum(axis=1)
    out["shared"] += (t & (nb >= 2)[None, :]).sum(axis=1)
    q = (np.uint64(Q32) // np.maximum(nb, 1).astype(np.uint64))
    out["share_q32"] += (t.astype(np.uint64) * q[None, :]).sum(axis=1, dtype=np.uint64)


def assign_loop(haps, rank, off, codes, max_mismatch=-1):
    """The same definition as a literal per-read Python loop (small inputs; checks ``assign``)."""
    H = len(haps)
    unique, shared, share = [0] * H, [0] * H, [0] * H
    tot = [0, 0, 0]
    best_mm, n_best, first_best = [], [], []
    for i in range(len(rank)):
        r, c = int(rank[i]), [int(x) for x in codes[off[i]:off[i + 1]]]
        inf = [t for t in range(len(c)) if c[t] not in (4, 6)]
        if not inf:
            tot[1] += 1
            best_mm.append(-1); n_best.append(0); first_best.append(-1)
            continue
        d = [sum(1 for t in inf if c[t] != int(haps[h][r + t + 1])) for h in range(H)]
        D = min(d)
        B = [h for h in range(H) if d[h] == D]
        best_mm.append(D); n_best.append(len(B))
        if max_mismatch >= 0 and D > max_mismatch:
            tot[2] += 1
            first_best.append(-1)
            continue
        tot[0] += 1
        first_best.append(B[0])
        for h in B:
            if len(B) == 1:
                unique[h] += 1
            else:
                shared[h] += 1
            share[h] += Q32 // len(B)
    return {"unique": np.array(unique, np.int64), "shared": np.array(shared, np.int64),
            "share_q32": np.array(share, np.uint64), "assigned": tot[0], "uninformative": tot[1],
            "over_limit": tot[2], "best_mm": np.array(best_mm, np.int32), "n_best": np.array(n_best, np.int32),
            "first_best": np.array(first_best, np.int32)}
