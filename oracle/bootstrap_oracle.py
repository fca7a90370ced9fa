"""Bootstrap of the abundance EM in numpy / plain Python, written from the definition in DESIGN.md §4 K8; the reference
has no counterpart.  Test infrastructure only: the product must not import it.

Inputs are K7's classes (class_off, members, count), H haplotypes, B replicates and a uint64 seed.  T = sum of count,
P[c] = sum of count[c'] over c' < c.  Replicate 0 is the EM on count.  Replicate b >= 1 draws T reads with
replacement, in pairs: for i = 0 .. ceil(T/2) - 1

    (x0, x1, x2, x3) = Philox4x32-10(counter = (lo32(i), hi32(i), b, 0), key = (lo32(seed), hi32(seed)))
    draw 2i   : x = x0 | x1 << 32
    draw 2i+1 : x = x2 | x3 << 32          (only if 2i+1 < T)
    u = floor(x * T / 2^64)                 (the high word of the 128-bit product)
    the draw lands in the class c with P[c] <= u < P[c+1];  count_b[c] = the draws that land in c

and runs K7's EM (abundance_oracle.em) on the classes with count_b >= 1, in class order, with the same T.
"""
from __future__ import annotations

import numpy as np

from oracle import abundance_oracle as ao

M0, M1 = 0xD2511F53, 0xCD9E8D57          # Philox4x32 multipliers
W0, W1 = 0x9E3779B9, 0xBB67AE85          # Weyl key increments
MASK32 = 0xFFFFFFFF
_M32 = np.uint64(MASK32)
_S32 = np.uint64(32)


def philox_scalar(ctr, key):
    """Philox4x32-10 of one counter (4 x uint32) and key (2 x uint32), with Python integers -> 4 x uint32."""
    c0, c1, c2, c3 = ctr
    k0, k1 = key
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & MASK32, (p0 >> 32) ^ c3 ^ k1, p0 & MASK32
    return c0, c1, c2, c3


def philox(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10, vectorised: uint32 values held in uint64 arrays (products of 32-bit halves fit) ->
    (x0, x1, x2, x3) as uint64 arrays of 32-bit values."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & _M32 for c in (c0, c1, c2, c3))
    k0, k1 = int(k0) & MASK32, int(k1) & MASK32
    m0, m1 = np.uint64(M0), np.uint64(M1)
    for r in range(10):
        if r:
            k0, k1 = (k0 + W0) & MASK32, (k1 + W1) & MASK32
        p0, p1 = m0 * c0, m1 * c2
        c0, c1, c2, c3 = ((p1 >> _S32) ^ c1 ^ np.uint64(k0), p1 & _M32, (p0 >> _S32) ^ c3 ^ np.uint64(k1),
                          p0 & _M32)
    return c0, c1, c2, c3


def mulhi(x, T):
    """floor(x * T / 2^64) for uint64 x (array) and 0 <= T < 2^64, by 32-bit limbs."""
    x = np.asarray(x, dtype=np.uint64)
    xl, xh = x & _M32, x >> _S32
    tl, th = np.uint64(int(T) & MASK32), np.uint64(int(T) >> 32)
    ll, lh, hl = xl * tl, xl * th, xh * tl
    mid = (ll >> _S32) + (lh & _M32) + (hl & _M32)
    return xh * th + (lh >> _S32) + (hl >> _S32) + (mid >> _S32)


def resample(count, seed, b, chunk_pairs=1 << 22):
    """count_b of replicate b >= 1 (int64 [C]), vectorised over chunks of draw pairs."""
    count = np.asarray(count, dtype=np.int64)
    T = int(count.sum())
    P = np.concatenate([[0], np.cumsum(count)]).astype(np.uint64)
    out = np.zeros(len(count), np.int64)
    n_pairs = (T + 1) // 2
    k0, k1 = int(seed) & MASK32, (int(seed) >> 32) & MASK32
    for a in range(0, n_pairs, chunk_pairs):
        i = np.arange(a, min(n_pairs, a + chunk_pairs), dtype=np.uint64)
        x0, x1, x2, x3 = philox(i & _M32, i >> _S32, np.full(len(i), b, np.uint64), np.zeros(len(i), np.uint64),
                                k0, k1)
        xa, xb = x0 | (x1 << _S32), x2 | (x3 << _S32)
        xb = xb[2 * i + 1 < np.uint64(T)]
        u = mulhi(np.concatenate([xa, xb]), T)
        c = np.searchsorted(P, u, side="right") - 1
        out += np.bincount(c, minlength=len(count)).astype(np.int64)
    return out


def resample_loop(count, seed, b):
    """The same draws as a literal per-draw Python loop (small T; checks ``resample``)."""
    count = [int(x) for x in count]
    T = sum(count)
    P = [0]
    for n in count:
        P.append(P[-1] + n)
    out = [0] * len(count)
    key = (seed & MASK32, (seed >> 32) & MASK32)
    for d in range(T):
        i = d // 2
        x = philox_scalar((i & MASK32, i >> 32, b, 0), key)
        v = x[0] | x[1] << 32 if d % 2 == 0 else x[2] | x[3] << 32
        u = v * T >> 64
        c = 0
        while not (P[c] <= u < P[c + 1]):
            c += 1
        out[c] += 1
    return np.array(out, np.int64)


def filtered(class_off, members, count_b):
    """The CSR of the classes with count_b >= 1, in class order."""
    keep = np.nonzero(np.asarray(count_b) >= 1)[0]
    size = np.diff(class_off)[keep]
    mem = np.concatenate([members[class_off[c]:class_off[c + 1]] for c in keep]) if len(keep) else np.zeros(0)
    return (np.concatenate([[0], np.cumsum(size)]).astype(np.int64), mem.astype(np.int32),
            np.asarray(count_b, np.int64)[keep])


def em_t(n_haps, class_off, members, count_b, T, max_iter=10000, tol=1e-12):
    """K7's EM on the filtered classes with the total T of the original counts (equal to the resampled total)."""
    o, m, n = filtered(class_off, members, count_b)
    assert int(n.sum()) == T
    return ao.em(n_haps, o, m, n, max_iter=max_iter, tol=tol)


def bootstrap(n_haps, class_off, members, count, n_boot, seed, max_iter=10000, tol=1e-12):
    """-> dict(pi float64 [B+1][H], n_iter, converged, loglik [B+1], count int64 [B+1][C])."""
    count = np.asarray(count, np.int64)
    T = int(count.sum())
    rows = [count] + [resample(count, seed, b) for b in range(1, n_boot + 1)]
    ems = [em_t(n_haps, class_off, members, r, T, max_iter, tol) for r in rows]
    return {"pi": np.array([e["pi"] for e in ems], np.float64).reshape(n_boot + 1, n_haps),
            "n_iter": np.array([e["n_iter"] for e in ems], np.int32),
            "converged": np.array([e["converged"] for e in ems], bool),
            "loglik": np.array([e["loglik"] for e in ems], np.float64),
            "count": np.stack(rows)}
