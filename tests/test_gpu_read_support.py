"""Read support on the GPU (hx_assign_reads / Hansel.assign_reads) against the numpy oracle of the definition
(oracle/support_oracle.py): every output, per read and per haplotype, must be equal."""
import gzip
import os

import numpy as np
import pytest

from gretel_b200 import _lib, bamio, synth, util
from gretel_b200.hansel import REF_SYMBOLS, REF_UNSYMBOLS, Hansel
from oracle import hansel_oracle as o
from oracle import support_oracle as so

pytestmark = pytest.mark.gpu

FIELDS = ("unique", "shared", "share_q32", "assigned", "uninformative", "over_limit", "best_mm", "n_best", "first_best")


def matrix(N):
    return Hansel.init_matrix(REF_SYMBOLS, REF_UNSYMBOLS, N, band_w=1, device=0)


def assert_same(got, exp):
    for f in FIELDS:
        assert np.array_equal(np.asarray(getattr(got, f)), np.asarray(exp[f])), f
    assert np.array_equal(got.share, exp["share_q32"].astype(np.float64) / 2.0 ** 32)


def check(h, haps, rank, off, codes, mm=-1):
    got = h.assign_reads(haps, rank, off, codes, max_mismatch=mm, per_read=True)
    exp = so.assign(haps, rank, off, codes, mm)
    assert_same(got, exp)
    assert got.assigned + got.uninformative + got.over_limit == len(rank)
    return got


def random_haps(rng, H, N, alphabet=7):
    haps = rng.integers(0, alphabet, size=(H, N + 1)).astype(np.uint8)
    haps[:, 0] = rng.integers(0, 256, size=H)           # site 0 is never read, whatever it holds
    return haps


def with_mutants(strains, H, rng, rate=0.02):
    """'_' + the strains, then copies of them with a fraction ``rate`` of the sites changed, H rows in all."""
    base = np.concatenate([np.full((len(strains), 1), 6, np.uint8), strains], axis=1)
    rows = [base[i % len(base)].copy() for i in range(H)]
    for i in range(len(base), H):
        hit = np.nonzero(rng.random(base.shape[1] - 1) < rate)[0] + 1
        rows[i][hit] = (rows[i][hit] + rng.integers(1, 4, size=len(hit))) % 4
    return np.stack(rows)


@pytest.mark.parametrize("mm", [-1, 0, 1, 3])
@pytest.mark.parametrize("H", [1, 2, 7, 33, 100, 300])
def test_adversarial_reads(H, mm):
    for seed in range(2):
        rng = np.random.default_rng(1000 * H + 10 * (mm + 1) + seed)
        N = int(rng.integers(40, 600))
        # a small alphabet on some haplotypes makes ties common
        haps = random_haps(rng, H, N, alphabet=7 if seed == 0 else 2)
        h = matrix(N)
        for sort in (True, False):
            rank, off, codes = synth.random_packed(rng, N, 3000, 40, p_special=0.2, sort=sort)
            check(h, haps, rank, off, codes, mm)


def geometry_reads(rng, N, ks):
    """Reads of every width in ks: from site 1, ending at site N, and first sites at every offset in a word."""
    rank, klen = [], []
    for k in ks:
        if k > N:
            continue
        starts = {0, N - k}
        for o in range(32):                         # first site r+1 at bit o of its word
            r = (o - 1) % 32
            if r <= N - k:
                starts.add(r)
        starts |= {int(x) for x in rng.integers(0, N - k + 1, size=8)}
        for r in sorted(starts):
            rank.append(r)
            klen.append(k)
    off = np.concatenate([[0], np.cumsum(klen)]).astype(np.int64)
    codes = rng.integers(0, 4, size=int(off[-1])).astype(np.uint8)
    sp = rng.random(len(codes)) < 0.1
    codes[sp] = rng.integers(4, 7, size=int(sp.sum()))
    return np.array(rank, np.int32), off, codes


@pytest.mark.parametrize("N", [31, 32, 33, 10_000])
def test_word_geometry(N):
    rng = np.random.default_rng(N)
    rank, off, codes = geometry_reads(rng, N, [1, 2, 31, 32, 33, 63, 64, 65, 300, 1000])
    assert (rank + np.diff(off) == N).any() and (rank == 0).any()
    h = matrix(N)
    for H, alphabet in ((5, 7), (9, 2)):
        haps = random_haps(rng, H, N, alphabet)
        # haplotypes that equal some reads exactly, so that d = 0 is reached at every width
        for j in range(min(H, 3)):
            i = int(rng.integers(0, len(rank)))
            haps[j, rank[i] + 1:rank[i] + 1 + np.diff(off)[i]] = codes[off[i]:off[i + 1]]
        for mm in (-1, 0, 2):
            check(h, haps, rank, off, codes, mm)


def test_duplicated_haplotype():
    rng = np.random.default_rng(5)
    N = 200
    x = random_haps(rng, 1, N)
    haps = np.concatenate([x, x])
    rank, off, codes = synth.random_packed(rng, N, 5000, 40, p_special=0.2)
    got = check(matrix(N), haps, rank, off, codes)
    assert got.assigned > 0
    assert got.unique.tolist() == [0, 0]
    assert got.shared.tolist() == [got.assigned] * 2
    assert got.share_q32.tolist() == [got.assigned * (1 << 31)] * 2
    assert (got.n_best[got.first_best >= 0] == 2).all()


def test_haplotypes_beyond_shared_memory():
    """More haplotypes than the per-CTA shared-memory sums hold: the rest are summed in global memory."""
    rng = np.random.default_rng(6)
    N = 64
    haps = random_haps(rng, 2500, N, alphabet=3)
    rank, off, codes = synth.random_packed(rng, N, 4000, 12, p_special=0.1, sort=False)
    got = check(matrix(N), haps, rank, off, codes)
    assert got.share_q32[2048:].sum() > 0


def test_chunked_input_equals_pieces_and_oracle():
    w = synth.scaled(synth.WORKLOADS["metagenome"], 2_200_000)
    d = synth.generate(w)
    rng = np.random.default_rng(7)
    haps = with_mutants(d["strains"], 8, rng)
    rank, off, codes = d["rank"], d["off"], d["codes"]
    assert len(rank) >= 2_000_000
    h = matrix(w.n_snps)
    whole = check(h, haps, rank, off, codes)
    cuts = [0, 123_457, 1_500_000, len(rank)]
    parts = [h.assign_reads(haps, rank[a:b], off[a:b + 1], codes, per_read=True) for a, b in zip(cuts[:-1], cuts[1:])]
    for f in ("unique", "shared", "share_q32"):
        assert np.array_equal(getattr(whole, f), sum(getattr(p, f) for p in parts)), f
    for f in ("assigned", "uninformative", "over_limit"):
        assert getattr(whole, f) == sum(getattr(p, f) for p in parts), f
    for f in ("best_mm", "n_best", "first_best"):
        assert np.array_equal(getattr(whole, f), np.concatenate([getattr(p, f) for p in parts])), f


def distinct_paths(paths):
    _, first = np.unique(paths, axis=0, return_index=True)
    return paths[np.sort(first)]


def test_recovered_haplotypes_hiv():
    w = synth.WORKLOADS["hiv"]
    d = synth.generate(w)
    N = w.n_snps
    rank, off, codes = d["rank"], d["off"], d["codes"]
    h = util.load_from_packed(rank, off, codes, N, band_w=d["max_k"] - 1, device=0)
    paths, _ = h.recover_codes(h.copy(), 10)
    haps = distinct_paths(paths)
    assert len(haps) >= 2
    band = h.band()
    got = check(h, haps, rank, off, codes)
    assert np.array_equal(h.band(), band), "assign_reads changed the matrix"
    assert h.kernel_ms("assign") > 0
    # the five true strains: reads go back to the strain they were drawn from
    strains = np.concatenate([np.full((5, 1), 6, np.uint8), d["strains"]], axis=1)
    got = check(h, strains, rank, off, codes)
    asg = got.first_best >= 0
    frac = float((got.first_best[asg] == d["strain_of"][asg]).mean())
    # observed 0.99975 (a read whose strains agree over all its sites goes to the lowest of them); margin 0.0028
    assert frac >= 0.997, frac
    emp = np.bincount(d["strain_of"], minlength=5) / len(rank)
    # observed within 6.6e-5 of the empirical read fractions; tolerance 1e-3
    assert np.abs(got.share / got.assigned - emp).max() <= 1e-3, (got.share / got.assigned, emp)


def test_long_reads():
    w = synth.scaled(synth.WORKLOADS["ont"], 5_000)
    d = synth.generate(w)
    assert d["max_k"] > 64
    haps = with_mutants(d["strains"], 20, np.random.default_rng(8), rate=0.05)
    h = matrix(w.n_snps)
    for mm in (-1, 20):
        check(h, haps, d["rank"], d["off"], d["codes"], mm)


def test_no_reads():
    h = matrix(10)
    haps = random_haps(np.random.default_rng(9), 3, 10)
    got = check(h, haps, np.zeros(0, np.int32), np.zeros(1, np.int64), np.zeros(0, np.uint8))
    assert got.unique.tolist() == [0, 0, 0] and got.share_q32.tolist() == [0, 0, 0]


def test_invalid_input_raises_and_leaves_handle_usable():
    rng = np.random.default_rng(10)
    N = 50
    h = matrix(N)
    haps = random_haps(rng, 4, N)
    rank, off, codes = synth.random_packed(rng, N, 500, 20)

    def expect(code, *args):
        with pytest.raises(_lib.HanselxError) as e:
            h.assign_reads(*args)
        assert e.value.code == code
        check(h, haps, rank, off, codes)                    # the handle still works

    past = np.concatenate([rank, [N - 1]]).astype(np.int32)  # a read of 2 sites from site N
    expect(_lib.HX_E_READ, haps, past, np.concatenate([off, [off[-1] + 2]]), np.concatenate([codes, [0, 1]]))
    bad = codes.copy()
    bad[len(bad) // 2] = 7
    expect(_lib.HX_E_READ, haps, rank, off, bad)
    bad_hap = haps.copy()
    bad_hap[2, 3] = 7
    expect(_lib.HX_E_ARG, bad_hap, rank, off, codes)
    expect(_lib.HX_E_ARG, haps[:0], rank, off, codes)


# ---- command line -----------------------------------------------------------------------------------------------
def expected_support(bam, vcf, contig, start, end, max_paths, max_mismatch=-1):
    """gretel.support as the oracle flow formats it: oracle recovery, distinct paths in i_0 order, oracle support."""
    v = bamio.process_vcf(vcf, contig, start, end)
    rank, off, codes = bamio.pack_bam(bam, contig, start, end, v)
    ho = o.load_from_packed(rank, off, codes, v["N"])
    _, PATHS = o.recover(ho, v["N"], max_paths=max_paths)
    keys = sorted(PATHS, key=lambda x: PATHS[x]["i_0"])
    haps = np.array([[REF_SYMBOLS.index(str(s)) for s in PATHS[k]["hansel_path"]] for k in keys], np.uint8)
    r = so.assign(haps, rank, off, codes, max_mismatch)
    lines = ["# %d\t%d\t%d\t%d\t%d" % (len(rank), r["assigned"], r["uninformative"], r["over_limit"], max_mismatch)]
    for j, k in enumerate(keys):
        share = int(r["share_q32"][j]) / 2.0 ** 32
        lines.append("%d\t%d\t%d\t%.2f\t%.4f" % (PATHS[k]["i_0"], r["unique"][j], r["shared"][j], share,
                                                 share / r["assigned"] if r["assigned"] else 0.0))
    return lines


def run_both(tmp_path, argv, extra):
    """The same run without and with --support: the same outputs, plus gretel.support."""
    from gretel_b200 import cmd
    plain, sup = tmp_path / "plain", tmp_path / "sup"
    plain.mkdir()
    sup.mkdir()
    assert cmd.main(argv + ["-o", str(plain)]) == 0
    assert cmd.main(argv + ["-o", str(sup), "--support"] + extra) == 0
    assert sorted(os.listdir(plain)) == ["gretel.crumbs", "out.fasta", "snp.fasta"]
    assert sorted(os.listdir(sup)) == ["gretel.crumbs", "gretel.support", "out.fasta", "snp.fasta"]
    for f in ("out.fasta", "snp.fasta", "gretel.crumbs"):
        assert (plain / f).read_bytes() == (sup / f).read_bytes(), f
    return open(sup / "gretel.support").read().split("\n")[:-1]


def test_cli_support_toy_bam(tmp_path, golden_dir):
    bam, vcf = os.path.join(golden_dir, "ref_test.bam"), os.path.join(golden_dir, "ref_test.vcf.gz")
    got = run_both(tmp_path, [bam, vcf, "hoot", "-s", "1", "-e", "20", "-p", "6", "--quiet"], [])
    assert got == expected_support(bam, vcf, "hoot", 1, 20, 6)


def synthetic_bam(tmp_path):
    """The BAM of test_gpu_cli.py::test_pipeline_on_synthetic_bam: 3 strains over 40 SNPs, 1500 reads with
    deletions."""
    from tests.bamwriter import write_bam
    rng = np.random.default_rng(123)
    G, N, R, L = 1200, 40, 1500, 100
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
        pos = int(rng.integers(0, G - L))
        if rng.random() < 0.15:
            cigar = [("M", 40), ("D", 3), ("M", L - 43)]
            seq = "".join(st[pos:pos + 40]) + "".join(st[pos + 43:pos + L])
        else:
            cigar = [("M", L)]
            seq = "".join(st[pos:pos + L])
        reads.append((0, pos, 0, "r%d" % i, cigar, seq))
    reads.sort(key=lambda r: r[1])
    bam, vcf = str(tmp_path / "s.bam"), str(tmp_path / "s.vcf.gz")
    write_bam(bam, [("ctg", G)], reads, block=20000)
    with gzip.open(vcf, "wt") as fh:
        fh.write("##fileformat=VCFv4.2\n")
        for p in sites:
            fh.write("ctg\t%d\t.\tA\tC,T,G\t0\t.\tINFO\n" % (p + 1))
    return bam, vcf, G


@pytest.mark.parametrize("max_mismatch", [-1, 1])
def test_cli_support_synthetic_bam(tmp_path, max_mismatch):
    bam, vcf, G = synthetic_bam(tmp_path)
    extra = ["--max-mismatch", str(max_mismatch)] if max_mismatch >= 0 else []
    got = run_both(tmp_path, [bam, vcf, "ctg", "-s", "1", "-e", str(G), "-p", "4", "--quiet", "-@", "2"], extra)
    exp = expected_support(bam, vcf, "ctg", 1, G, 4, max_mismatch)
    assert got == exp
    assert len(exp) >= 3
