"""Path scores written from the definition in DESIGN.md (§4 K6): the branch weights of Hansel.get_edge_weights_at at
every site of a given haplotype; the reference has no counterpart.  Test infrastructure only: the product must not
import it.

For haplotype p (p[0] = '_', codes 0..6 at sites 1..N) and site s in 1..N: w[s] = get_edge_weights_at(s, p[0..s-1])
with the matrix's L and flags, normalised (0 for a non-candidate), plus its total; best[s] = the first maximum over the
candidates in symbol order (gretel.py:159-174), 255 where there is none; w_hap[s] = w[s][p[s]] (0 if p[s] is not a
candidate); w_second[s] = the largest weight of the candidates other than p[s] (0 if none).  Per haplotype: loglik =
sum of log10(w_hap) over the sites with w_hap > 0, in site order; n_unsupported = sites with w_hap == 0; n_disagree =
sites with best != p[s].

``score`` applies it through OracleHansel.get_edge_weights_at (the literal Python restatement), ``score_c`` through
or_edge_weights_at of the C twin on the banded layout (full-size checks).
"""
from __future__ import annotations

from math import log10

import numpy as np

from . import hansel_oracle as ho

NO_CANDIDATE = 255


def _empty(H, N):
    """The outputs of H haplotypes over N sites, zeroed."""
    out = {"weights": np.zeros((H, N, 8)), "w_hap": np.zeros((H, N)), "w_second": np.zeros((H, N)),
           "best": np.zeros((H, N), np.uint8), "loglik": np.zeros(H), "n_unsupported": np.zeros(H, np.int32),
           "n_disagree": np.zeros(H, np.int32)}
    return out


def _site(out, h, s, a, w, mask):
    """Fill site s (1-based) of haplotype h: allele a, weights w[7] (0 for non-candidates), candidate mask."""
    best = -1
    for q in range(7):                                       # gretel.py:166-174: the first maximum
        if mask >> q & 1 and (best < 0 or w[q] > w[best]):
            best = q
    out["best"][h, s - 1] = NO_CANDIDATE if best < 0 else best
    out["w_hap"][h, s - 1] = w[a] if mask >> a & 1 else 0.0
    out["w_second"][h, s - 1] = max([w[q] for q in range(7) if mask >> q & 1 and q != a], default=0.0)


def _sums(out, paths):
    for h in range(paths.shape[0]):
        ll, unsup, dis = 0.0, 0, 0
        for s in range(1, paths.shape[1]):
            wh = float(out["w_hap"][h, s - 1])
            if wh > 0:
                ll += log10(wh)
            else:
                unsup += 1
            dis += int(out["best"][h, s - 1]) != int(paths[h, s])
        out["loglik"][h], out["n_unsupported"][h], out["n_disagree"][h] = ll, unsup, dis
    return out


def check_paths(paths, N):
    paths = np.asarray(paths, dtype=np.uint8)
    if paths.ndim != 2 or paths.shape[1] != N + 1:
        raise ValueError("paths must be [H][N+1]")
    if (paths[:, 0] != 6).any() or (paths > 6).any():
        raise ValueError("a path must hold '_' at site 0 and codes 0..6")
    return paths


def score(hansel, paths, L=None):
    """Through OracleHansel.get_edge_weights_at (``hansel``: an OracleHansel; L defaults to hansel.L)."""
    N = hansel.n_snps
    paths = check_paths(paths, N)
    saved = hansel.L
    hansel.L = saved if L is None else L
    try:
        H = paths.shape[0]
        out = _empty(H, N)
        for h in range(H):
            sym = [ho.SYMBOLS[c] for c in paths[h]]
            for s in range(1, N + 1):
                br = hansel.get_edge_weights_at(s, sym)
                mask, w = 0, [0.0] * 7
                for q, name in enumerate(ho.SYMBOLS):
                    if name in br:
                        mask |= 1 << q
                        w[q] = br[name]
                out["weights"][h, s - 1, :7] = w
                out["weights"][h, s - 1, 7] = br["total"]
                _site(out, h, s, int(paths[h, s]), w, mask)
    finally:
        hansel.L = saved
    return _sums(out, paths)


def score_c(c_oracle, band_f32, N, W, L, paths, v_site="from", skip_unsym=True):
    """Through or_edge_weights_at of the C twin, site by site (band float32 [N+2][W][7][7])."""
    paths = check_paths(paths, N)
    H = paths.shape[0]
    out = _empty(H, N)
    for h in range(H):
        p = np.ascontiguousarray(paths[h])
        for s in range(1, N + 1):
            mask, w, tw = c_oracle.edge_weights_at(band_f32, N, W, L, s, p, v_site, skip_unsym)
            out["weights"][h, s - 1, :7] = w
            out["weights"][h, s - 1, 7] = tw
            _site(out, h, s, int(p[s]), w, mask)
    return _sums(out, paths)
