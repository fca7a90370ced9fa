"""The path-score oracle (oracle/score_oracle.py) by hand on the reference's golden toy, and its literal Python form
(OracleHansel.get_edge_weights_at per site) against the C twin (or_edge_weights_at per site) on random matrices.
Codes: A0 C1 G2 T3 N4 -5 _6."""
import os

import numpy as np
import pytest

from gretel_b200 import bamio, synth
from oracle import hansel_oracle as o
from oracle import score_oracle as so

A, C, G, T, N, DEL, GAP = range(7)
FIELDS = ("weights", "w_hap", "w_second", "best", "loglik", "n_unsupported", "n_disagree")


def toy(golden_dir):
    v = bamio.process_vcf(os.path.join(golden_dir, "ref_test.vcf.gz"), "hoot", 1, 19)
    rank, off, codes = bamio.pack_bam(os.path.join(golden_dir, "ref_test.bam"), "hoot", 1, 19, v)
    return o.load_from_packed(rank, off, codes, v["N"])


def same(a, b):
    for f in FIELDS:
        assert np.array_equal(np.asarray(a[f]), np.asarray(b[f])), f


def test_toy_site_one_by_hand(golden_dir):
    """Site 1 of the toy: counts A1 C1 T2 (total 4); the only lookback is the start sentinel, where '_' precedes
    A once, C once and T twice and no valid symbol is seen (V = 0), so the terms are (1+1)/1, (1+1)/1, (1+2)/2.
    Weights 1/4*2, 1/4*2, 2/4*3/2 = 0.5, 0.5, 0.75; total 1.75; normalised 2/7, 2/7, 3/7: T is the pick."""
    h = toy(golden_dir)
    assert h.n_snps == 3 and h.L == 3
    paths = np.array([[GAP, T, T, G], [GAP, A, T, G], [GAP, G, T, G], [GAP, N, T, G]], np.uint8)
    r = so.score(h, paths)
    w1 = r["weights"][:, 0]
    for row in w1:
        assert row[[A, C, T]] == pytest.approx([2 / 7, 2 / 7, 3 / 7], rel=1e-15)
        assert row[[G, N, DEL, GAP]].tolist() == [0.0] * 4
        assert row[7] == pytest.approx(1.75, rel=1e-15)
    assert r["best"][:, 0].tolist() == [T] * 4
    assert r["w_hap"][:, 0].tolist() == [w1[0][T], w1[1][A], 0.0, 0.0]       # G unseen; N is not a candidate
    assert r["w_second"][:, 0].tolist() == [w1[0][A], w1[1][T], w1[2][T], w1[3][T]]
    # site 1 is the only disagreement of the second path; the third and fourth are unsupported there
    assert r["n_disagree"][1] >= 1 and r["n_unsupported"][2] >= 1 and r["n_unsupported"][3] >= 1
    for k in range(4):
        ll = 0.0
        for s in range(3):
            if r["w_hap"][k, s] > 0:
                ll += np.log10(r["w_hap"][k, s])
        assert r["loglik"][k] == pytest.approx(ll, rel=1e-15)
        assert r["n_unsupported"][k] == int((r["w_hap"][k] == 0).sum())
        assert r["n_disagree"][k] == int((r["best"][k] != paths[k, 1:]).sum())


def test_toy_recovered_path_agrees_everywhere(golden_dir):
    """The walk picks `best` at every site, so its own path scores n_disagree = 0 on the matrix it walked."""
    h = toy(golden_dir)
    path, _, _ = o.generate_path(h.n_snps, h, h.copy())
    codes = np.array([[o.CODE[s] for s in path]], np.uint8)
    r = so.score(h, codes)
    assert r["n_disagree"].tolist() == [0] and r["n_unsupported"].tolist() == [0]
    assert r["best"][0].tolist() == codes[0, 1:].tolist()


def test_bad_paths_are_refused(golden_dir):
    h = toy(golden_dir)
    with pytest.raises(ValueError):
        so.score(h, np.array([[A, T, T, G]], np.uint8))
    with pytest.raises(ValueError):
        so.score(h, np.array([[GAP, 7, T, G]], np.uint8))


def random_case(seed, n_snps=11, n_reads=60, max_k=6):
    rng = np.random.default_rng(seed)
    rank, off, codes = synth.random_packed(rng, n_snps, n_reads, max_k, p_special=0.15)
    return rng, rank, off, codes


@pytest.mark.parametrize("L", range(1, 9))
@pytest.mark.parametrize("v_site,skip", [("from", True), ("to", True), ("from", False), ("to", False)])
def test_python_and_c_agree(c_oracle, L, v_site, skip):
    rng, rank, off, codes = random_case(100 * L + 2 * (v_site == "to") + skip)
    n = 11
    h = o.load_from_packed(rank, off, codes, n, v_site=v_site, candidates_skip_unsymbols=skip)
    paths = rng.integers(0, 7, size=(4, n + 1)).astype(np.uint8)
    paths[:, 0] = GAP
    paths[0, 1:] = rng.integers(0, 4, size=n)                 # one path of plain alleles
    for W in (n + 1, 3):                                      # the whole triangle, and terms beyond a narrow band
        band = o.band_of(h, W)
        if W < n + 1:                                         # what a W-wide band keeps of the matrix
            hb = h.copy()
            hb.m[...] = 0
            for pj in range(1, n + 2):
                for d in range(1, W + 1):
                    if pj - d >= 0:
                        hb.m[:, :, pj - d, pj] = h.m[:, :, pj - d, pj]
        else:
            hb = h
        exp = so.score(hb, paths, L=L)
        got = so.score_c(c_oracle, band, n, W, L, paths, v_site, skip)
        same(got, exp)
