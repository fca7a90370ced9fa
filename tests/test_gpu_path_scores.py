"""Path scores on the GPU (hx_score_paths / Hansel.score_paths, DESIGN.md §4 K6) against the oracle of the definition
(oracle/score_oracle.py: the literal Python one and its C twin), with no tolerance: every weight, pick and sum must be
equal.  Both term paths of k_score_sites (the walk tables, and the terms read from the band) are forced in turn with
HX_SCORE_TABLES and must give the same bytes.  A path the walk chose must score n_disagree = 0 against the matrix
the walk saw."""
import contextlib
import gzip
import os

import numpy as np
import pytest

from gretel_b200 import _lib, bamio, synth, util
from gretel_b200.hansel import REF_SYMBOLS, REF_UNSYMBOLS, Hansel
from oracle import hansel_oracle as o
from oracle import score_oracle as so

pytestmark = pytest.mark.gpu

A, C, G, T, N_, DEL, GAP = range(7)
FIELDS = ("weights", "w_hap", "w_second", "best", "loglik", "n_unsupported", "n_disagree")
FLAGS = [("from", True), ("to", True), ("from", False), ("to", False)]


@contextlib.contextmanager
def env(**kw):
    old = {k: os.environ.get(k) for k in kw}
    for k, v in kw.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def device(band, N, W, L, v_site="from", skip=True):
    h = Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=W, device=0)
    h.load_band(band)
    h.L, h.v_site, h.candidates_skip_unsymbols = L, v_site, skip
    return h


def gpu(h, paths, tables=None, L=None, scratch_mb=None):
    with env(HX_SCORE_TABLES=None if tables is None else int(tables), HX_SCORE_SCRATCH_MB=scratch_mb):
        r = h.score_paths(paths, L=L, weights=True)
    return {f: getattr(r, f) for f in FIELDS}


def same(got, exp, what=""):
    for f in FIELDS:
        g, e = np.asarray(got[f]), np.asarray(exp[f])
        assert g.shape == e.shape, (what, f)
        bad = np.argwhere(g != e)
        assert bad.size == 0, "%s %s differs at %s: %r != %r" % (what, f, bad[0], g[tuple(bad[0])], e[tuple(bad[0])])


def both_paths(h, paths, exp, L=None, scratch_mb=None, what=""):
    """Tables forced on and off: each equals the oracle, and the two give identical bytes."""
    a = gpu(h, paths, True, L, scratch_mb)
    b = gpu(h, paths, False, L, scratch_mb)
    same(a, exp, what + " tables")
    same(b, exp, what + " band")
    for f in FIELDS:
        assert np.asarray(a[f]).tobytes() == np.asarray(b[f]).tobytes(), (what, f)
    return a


def random_band(c_oracle, rng, N, n_reads, max_k, p_special=0.15):
    rank, off, codes = synth.random_packed(rng, N, n_reads, max_k, p_special=p_special)
    band, _ = c_oracle.ingest(rank, off, codes, N, max(1, max_k - 1))
    return band.astype(np.float32)


def random_paths(rng, H, N, special=True):
    p = rng.integers(0, 7 if special else 4, size=(H, N + 1)).astype(np.uint8)
    p[:, 0] = GAP
    return p


# ---- against the oracle ----------------------------------------------------------------------------------------------
def test_golden_toy(golden_dir):
    v = bamio.process_vcf(os.path.join(golden_dir, "ref_test.vcf.gz"), "hoot", 1, 19)
    rank, off, codes = bamio.pack_bam(os.path.join(golden_dir, "ref_test.bam"), "hoot", 1, 19, v)
    ho = o.load_from_packed(rank, off, codes, v["N"])
    N = v["N"]
    paths = np.array([[GAP, T, A, C], [GAP, A, C, A], [GAP, G, T, G], [GAP, N_, DEL, GAP], [GAP, T, T, C]], np.uint8)
    exp = so.score(ho, paths)
    h = device(o.band_of(ho, N + 1), N, N + 1, ho.L)
    got = both_paths(h, paths, exp, what="toy")
    assert (got["best"][:, 0] == T).all()                 # site 1: T 3/7 against A and C at 2/7 each (by hand)
    assert got["w_hap"][2, 0] == 0.0 and got["n_unsupported"][2] == 3


@pytest.mark.parametrize("L", range(1, 9))
@pytest.mark.parametrize("v_site,skip", FLAGS)
def test_random_matrices_every_lookback(c_oracle, L, v_site, skip):
    """N = 37 (not a multiple of the 4 items per warp), haplotypes with N, - and _; W = 5 so that L > W has terms
    beyond the band, and L > s near the start."""
    rng = np.random.default_rng(1000 * L + 10 * (v_site == "to") + skip)
    N, max_k = 37, 6
    band = random_band(c_oracle, rng, N, 300, max_k)
    paths = random_paths(rng, 6, N)
    paths[0, 1:] = rng.integers(0, 4, size=N)
    exp = so.score_c(c_oracle, band, N, max_k - 1, L, paths, v_site, skip)
    h = device(band, N, max_k - 1, L, v_site, skip)
    both_paths(h, paths, exp, what="L%d" % L)
    same(gpu(h, paths), exp, "default path")


@pytest.mark.parametrize("N", [1, 2, 3, 5, 6])
def test_tiny_regions(c_oracle, N):
    rng = np.random.default_rng(70 + N)
    band = random_band(c_oracle, rng, N, 40, min(N, 3) + 1)
    W = max(1, min(N, 3))
    for L in (1, 3, 8):
        paths = random_paths(rng, 5, N)
        exp = so.score_c(c_oracle, band, N, W, L, paths)
        both_paths(device(band, N, W, L), paths, exp, what="N%d L%d" % (N, L))


@pytest.mark.parametrize("H", [1, 40])
def test_scratch_chunks(c_oracle, H):
    """One haplotype, and 40 in chunks: a 1 MB scratch budget holds fewer than 40 haplotypes of 1500 sites (and less
    than the tables), so the haplotypes go through in several chunks on both paths."""
    rng = np.random.default_rng(90 + H)
    N, max_k, L = 1500, 9, 6
    band = random_band(c_oracle, rng, N, 3000, max_k)
    paths = random_paths(rng, H, N)
    sub = [0, H - 1]
    exp_sub = so.score_c(c_oracle, band, N, max_k - 1, L, paths[sub])
    h = device(band, N, max_k - 1, L)
    whole = gpu(h, paths, True)
    for mb in (1, 3):
        chunked = both_paths(h, paths, whole, scratch_mb=mb, what="%d MB" % mb)
        same({f: np.asarray(chunked[f])[sub] for f in FIELDS}, exp_sub, "chunked vs oracle")


def test_unobserved_allele_and_site_without_candidate(c_oracle):
    """An allele never seen at a site scores w_hap = 0 (counted in n_unsupported); a site with no counts at all has
    no candidate: best = 255, w_hap = w_second = 0."""
    rng = np.random.default_rng(5)
    N, max_k, L = 30, 6, 4
    rank, off, codes = synth.random_packed(rng, N, 200, max_k, p_special=0.0)
    codes[:] = np.where(codes == G, A, codes)                 # G is never observed
    band, _ = c_oracle.ingest(rank, off, codes, N, max_k - 1)
    band = band.astype(np.float32)
    hole = 12
    band[hole + 1, 0] = 0                                     # cell (12, 13): no counts at site 12
    paths = random_paths(rng, 3, N, special=False)
    paths[1, 1:] = G
    exp = so.score_c(c_oracle, band, N, max_k - 1, L, paths)
    got = both_paths(device(band, N, max_k - 1, L), paths, exp, what="holes")
    assert (got["best"][:, hole - 1] == 255).all() and (got["w_hap"][:, hole - 1] == 0).all()
    assert (got["w_second"][:, hole - 1] == 0).all()
    assert got["n_unsupported"][1] == N and got["loglik"][1] == 0.0


def test_config3_size_against_c_oracle(c_oracle):
    """N = 10k sites of the config-3 metagenome (1M reads): 10 recovered haplotypes and the 5 true strains, scored on
    the matrix before recovery."""
    w = synth.scaled(synth.WORKLOADS["metagenome"], 1_000_000)
    d = synth.generate(w)
    N, W = w.n_snps, d["max_k"] - 1
    h = util.load_from_packed(d["rank"], d["off"], d["codes"], N, band_w=W)
    assert h.L <= 32 and h.L <= W
    band = h.band()
    work = h.copy()
    paths, _ = work.recover_codes(h, 10, 0.01)
    assert len(paths) == 10
    strains = np.concatenate([np.full((5, 1), GAP, np.uint8), d["strains"]], axis=1)
    allp = np.concatenate([paths, strains])
    exp = so.score_c(c_oracle, band, N, W, h.L, allp)
    got = both_paths(h, allp, exp, what="config 3")
    assert got["n_disagree"][0] == 0                      # the first haplotype was walked on this matrix
    assert np.array_equal(h.band(), band)


def ont_region(n_reads=6000, n_sites=2000, max_k=400):
    """ONT-like reads (synth 'ont') cut to its first n_sites sites and to at most max_k sites each: L ~ 290.  Reads
    that run past site n_sites end there, so the end sentinel is counted and the last site has candidates."""
    w = synth.scaled(synth.WORKLOADS["ont"], n_reads)
    d = synth.generate(w)
    rank = d["rank"].astype(np.int64)
    k = np.minimum(np.minimum(np.diff(d["off"]), n_sites - rank), max_k)
    keep = (rank < n_sites) & (k >= 2)
    off = np.concatenate([[0], np.cumsum(k[keep])]).astype(np.int64)
    codes = np.concatenate([d["codes"][a:a + n] for a, n in zip(d["off"][:-1][keep], k[keep])]).astype(np.uint8)
    h = util.load_from_packed(rank[keep].astype(np.int32), off, codes, n_sites, band_w=max_k - 1)
    return h, d["strains"][:, :n_sites]


def test_ont_width_against_c_oracle(c_oracle):
    """L ~ 290 (the k_walk_wide regime): the default is the band path; the tables are forced too."""
    h, strains = ont_region()
    N, W, L = h.n_snps, h.band_w, h.L
    assert L > 200 and L <= W
    band = h.band()
    work = h.copy()
    paths, _ = work.recover_codes(h, 2, 0.01)
    assert len(paths) == 2
    allp = np.concatenate([paths, np.concatenate([np.full((2, 1), GAP, np.uint8), strains[:2]], axis=1)])
    exp = so.score_c(c_oracle, band, N, W, L, allp)
    got = both_paths(h, allp, exp, what="ont")
    same(gpu(h, allp), exp, "ont default")
    assert got["n_disagree"][0] == 0


# ---- against the single-site entry point ---------------------------------------------------------------------------
def test_weights_equal_get_edge_weights_at(c_oracle):
    rng = np.random.default_rng(9)
    N, max_k = 300, 8
    band = random_band(c_oracle, rng, N, 1500, max_k)
    for v_site, skip in FLAGS:
        h = device(band, N, max_k - 1, 5, v_site, skip)
        paths = random_paths(rng, 4, N)
        got = gpu(h, paths)
        for hh, s in zip(rng.integers(0, 4, 40), rng.integers(1, N + 1, 40)):
            ref = h.get_edge_weights_at(int(s), h.decode_path(paths[hh]))
            w = got["weights"][hh, s - 1]
            assert w[7] == ref["total"]
            for q, name in enumerate(REF_SYMBOLS):
                assert w[q] == ref.get(name, 0.0), (hh, s, name)


# ---- against the walk -----------------------------------------------------------------------------------------------
def walk_and_score(h, n, L=None):
    """generate_path_codes + reweight_path_codes one haplotype at a time; every path is scored on the matrix right
    before its reweight.  -> the scores of the paths."""
    orig = h.copy()
    out = []
    for _ in range(n):
        r = h.generate_path_codes(orig, L=L)
        assert r[0] is not None, "a hole at %d" % r[1]
        sc = h.score_paths(r[0][None, :], L=L)
        assert sc.n_disagree[0] == 0 and sc.n_unsupported[0] == 0
        assert np.array_equal(sc.best[0], r[0][1:])
        out.append(sc)
        h.reweight_path_codes(r[0], max(r[3], 0.01))
    return out


def thin(c_oracle, seed, N, max_k=40):
    rng = np.random.default_rng(seed)
    rank, off, codes = synth.random_packed(rng, N, 6 * N, max_k, p_special=0.05)
    rank = np.concatenate([rank, np.array([0, N - max_k], np.int32)])
    off = np.concatenate([off, off[-1] + max_k * np.arange(1, 3)])
    codes = np.concatenate([codes, rng.integers(0, 4, 2 * max_k).astype(np.uint8)])
    band, _ = c_oracle.ingest(rank, off, codes, N, max_k - 1)
    return band.astype(np.float32)


@pytest.mark.parametrize("tables", [True, False])
def test_walk_sequential(c_oracle, tables):
    N = 700
    with env(HX_SCORE_TABLES=int(tables)):
        walk_and_score(device(thin(c_oracle, 31, N), N, 39, 7), 5)


@pytest.mark.parametrize("L", [6, 20])
def test_walk_in_blocks_where_speculation_fails(c_oracle, L):
    """N >= 1024, L <= 32: the parallel-in-time walk, on two strains that differ at every site (blocks whose guessed
    history is the other strain are walked again)."""
    from tests.test_gpu_walk_blocks import MAX_K, strain_band
    band, _ = strain_band(c_oracle, 300 + L, 2400, 2, 3 * 2400)
    with env(HX_SCORE_TABLES=1):
        walk_and_score(device(band, 2400, MAX_K - 1, L), 4)
    with env(HX_SCORE_TABLES=0):
        walk_and_score(device(band, 2400, MAX_K - 1, L), 2)


def test_walk_beyond_fixed_point(c_oracle):
    """L = 36 > 32 (k_walk_tables) on a thin band, and ONT width (k_walk_wide)."""
    N = 1200
    walk_and_score(device(thin(c_oracle, 77, N), N, 39, 36), 3)
    h, _ = ont_region(n_reads=3000, n_sites=1200)
    walk_and_score(h, 2)


# ---- side effects and errors ----------------------------------------------------------------------------------------
def test_matrix_untouched_and_bad_paths(c_oracle):
    rng = np.random.default_rng(3)
    N, max_k = 200, 7
    h = device(random_band(c_oracle, rng, N, 800, max_k), N, max_k - 1, 4)
    before = h.band().tobytes()
    counts = [h.get_counts_at(i) for i in range(N + 1)]
    gpu(h, random_paths(rng, 5, N), True)
    gpu(h, random_paths(rng, 5, N), False)
    assert h.kernel_ms("score") > 0
    assert h.band().tobytes() == before
    h._touch()
    assert [h.get_counts_at(i) for i in range(N + 1)] == counts
    bad = random_paths(rng, 3, N)
    bad[2, 100] = 7
    with pytest.raises(_lib.HanselxError) as e:
        h.score_paths(bad)
    assert e.value.code == _lib.HX_E_ARG
    bad = random_paths(rng, 3, N)
    bad[1, 0] = A
    with pytest.raises(_lib.HanselxError) as e:
        h.score_paths(bad)
    assert e.value.code == _lib.HX_E_ARG
    assert h.band().tobytes() == before


# ---- CLI --------------------------------------------------------------------------------------------------------------
def expected_lines(ho, vcf_h, keyed):
    """gretel.scores / gretel.sites rows from the oracle: keyed = [(key, path codes)]."""
    paths = np.stack([p for _, p in keyed])
    r = so.score(ho, paths)
    scores, sites = [], []
    for j, (k, p) in enumerate(keyed):
        scores.append("%s\t%r\t%d\t%d" % (k, float(r["loglik"][j]), r["n_unsupported"][j], r["n_disagree"][j]))
        for s in range(1, vcf_h["N"] + 1):
            b = int(r["best"][j, s - 1])
            sites.append("%s\t%d\t%d\t%s\t%r\t%s\t%r\t%r" % (
                k, s, vcf_h["snp_rev"][s - 1], REF_SYMBOLS[p[s]], float(r["w_hap"][j, s - 1]),
                "." if b == 255 else REF_SYMBOLS[b], 0.0 if b == 255 else float(r["weights"][j, s - 1, b]),
                float(r["w_second"][j, s - 1])))
    return scores, sites


def run_cli(tmp_path, name, argv):
    from gretel_b200 import cmd
    out = tmp_path / name
    out.mkdir()
    assert cmd.main(argv + ["-o", str(out), "--quiet"]) == 0
    return out


def check_cli(tmp_path, bam, vcf, contig, end, n_paths, fasta, records):
    base = [bam, vcf, contig, "-s", "1", "-e", str(end), "-p", str(n_paths), "--support"]
    plain = run_cli(tmp_path, "plain", base)
    scored = run_cli(tmp_path, "scored", base + ["--site-weights", "--score", fasta])
    for f in ("out.fasta", "snp.fasta", "gretel.crumbs", "gretel.support"):
        assert (plain / f).read_bytes() == (scored / f).read_bytes(), f
    assert not (plain / "gretel.scores").exists() and not (plain / "gretel.sites").exists()
    v = bamio.process_vcf(vcf, contig, 1, end)
    rank, off, codes = bamio.pack_bam(bam, contig, 1, end, v)
    ho = o.load_from_packed(rank, off, codes, v["N"])
    _, PATHS = o.recover(ho.copy(), v["N"], max_paths=n_paths)
    keyed = [(PATHS[k]["i_0"], np.array([o.CODE[x] for x in PATHS[k]["hansel_path"]], np.uint8))
             for k in sorted(PATHS, key=lambda x: PATHS[x]["i_0"])]
    from gretel_b200 import gretel
    keyed += [(name, gretel.sequence_path(seq, v)) for name, seq in records]
    exp_scores, exp_sites = expected_lines(ho, v, keyed)
    got_scores = (scored / "gretel.scores").read_text().strip().split("\n")
    got_sites = (scored / "gretel.sites").read_text().strip().split("\n")
    assert got_scores[0].startswith("#") and got_sites[0].startswith("#")
    assert got_scores[1:] == exp_scores
    assert got_sites[1:] == exp_sites
    only = run_cli(tmp_path, "score_only", base + ["--score", fasta])
    assert (only / "gretel.scores").read_bytes() == (scored / "gretel.scores").read_bytes()
    assert not (only / "gretel.sites").exists()
    return {row.split("\t")[0]: row.split("\t") for row in got_scores[1:]}


def test_cli_toy(tmp_path, golden_dir):
    bam, vcf = os.path.join(golden_dir, "ref_test.bam"), os.path.join(golden_dir, "ref_test.vcf.gz")
    records = [("known", "TAAAAAAAAGAAAAAAAAA"), ("other", "ACGT")]
    fasta = tmp_path / "known.fasta"
    fasta.write_text("".join(">%s description\n%s\n" % r for r in records))
    check_cli(tmp_path, bam, vcf, "hoot", 19, 6, str(fasta), records)


def test_cli_synthetic_strains(tmp_path):
    """Three strains over 40 SNPs: the dominant one is recovered first, so it scores n_disagree = 0 and the loglik
    of haplotype 0."""
    from tests.bamwriter import write_bam
    rng = np.random.default_rng(123)
    G, N, R, RL = 1200, 40, 1500, 100
    sites = 20 + np.cumsum(rng.integers(5, 50, size=N))
    ref = rng.choice(list("ACGT"), size=G)
    strains = []
    for s in range(3):
        g = ref.copy()
        for p in sites:
            if rng.random() < 0.6:
                g[p] = rng.choice([b for b in "ACGT" if b != ref[p]])
        strains.append(g)
    reads = []
    for i in range(R):
        st = strains[rng.choice(3, p=[0.5, 0.3, 0.2])]
        pos = int(rng.integers(0, G - RL))
        reads.append((0, pos, 0, "r%d" % i, [("M", RL)], "".join(st[pos:pos + RL])))
    reads.sort(key=lambda r: r[1])
    bam, vcf = str(tmp_path / "s.bam"), str(tmp_path / "s.vcf.gz")
    write_bam(bam, [("ctg", G)], reads, block=20000)
    with gzip.open(vcf, "wt") as fh:
        fh.write("##fileformat=VCFv4.2\n")
        for p in sites:
            fh.write("ctg\t%d\t.\tA\tC,T,G\t0\t.\tINFO\n" % (p + 1))
    records = [("strain%d" % s, "".join(strains[s]).lower() if s == 2 else "".join(strains[s])) for s in range(3)]
    fasta = tmp_path / "strains.fasta"
    fasta.write_text("".join(">%s\n%s\n%s\n" % (n, s[:600], s[600:]) for n, s in records))
    rows = check_cli(tmp_path, bam, vcf, "ctg", G, 4, str(fasta), records)
    assert rows["strain0"][3] == "0"
    assert rows["strain0"][1] == rows["0"][1]
