"""Read classes on the GPU (hx_read_classes / Hansel.read_classes) against the numpy oracle of the definition
(oracle/abundance_oracle.py): the CSR arrays and totals must be equal, and the class sums must equal read support
(hx_assign_reads) on the same input.  Then the EM over GPU classes against the oracle's EM, bit for bit, and against
known abundances; and gretel.abundance on the command line."""
import os

import numpy as np
import pytest

from gretel_b200 import _lib, bamio, synth, util
from gretel_b200.hansel import REF_SYMBOLS, em_abundance
from oracle import abundance_oracle as ao
from oracle import hansel_oracle as o
from tests.test_gpu_read_support import geometry_reads, matrix, random_haps, synthetic_bam, with_mutants

pytestmark = pytest.mark.gpu

Q = 1 << 32


def class_sums(cls, H):
    """unique, shared and share_q32 per haplotype from CSR classes."""
    size = np.diff(cls.class_off)
    of = np.repeat(np.arange(len(cls.count)), size)
    n, s = cls.count[of], size[of]
    unique = np.bincount(cls.members[s == 1], weights=n[s == 1], minlength=H).astype(np.int64)
    shared = np.bincount(cls.members[s >= 2], weights=n[s >= 2], minlength=H).astype(np.int64)
    share = np.zeros(H, np.uint64)
    np.add.at(share, cls.members, n.astype(np.uint64) * (np.uint64(Q) // s.astype(np.uint64)))
    return unique, shared, share


def check(h, haps, rank, off, codes, mm=-1):
    got = h.read_classes(haps, rank, off, codes, max_mismatch=mm)
    exp = ao.classes(haps, rank, off, codes, mm)
    for k in ("class_off", "members", "count"):
        assert np.array_equal(getattr(got, k), exp[k]), k
    for k in ("assigned", "uninformative", "over_limit"):
        assert getattr(got, k) == exp[k], k
    sup = h.assign_reads(haps, rank, off, codes, max_mismatch=mm)
    unique, shared, share = class_sums(got, len(haps))
    assert np.array_equal(unique, sup.unique)
    assert np.array_equal(shared, sup.shared)
    assert np.array_equal(share, sup.share_q32)
    assert int(got.count.sum()) == got.assigned == sup.assigned
    assert (got.uninformative, got.over_limit) == (sup.uninformative, sup.over_limit)
    return got


@pytest.mark.parametrize("mm", [-1, 0, 1, 3])
@pytest.mark.parametrize("H", [1, 2, 7, 33, 100, 300])
def test_grid(H, mm):
    for alphabet in (7, 2):
        rng = np.random.default_rng(1000 * H + 10 * (mm + 1) + alphabet)
        N = int(rng.integers(40, 600))
        haps = random_haps(rng, H, N, alphabet=alphabet)
        h = matrix(N)
        for sort in (True, False):
            rank, off, codes = synth.random_packed(rng, N, 3000, 40, p_special=0.2, sort=sort)
            check(h, haps, rank, off, codes, mm)


@pytest.mark.parametrize("N", [31, 32, 33, 10_000])
def test_word_geometry(N):
    rng = np.random.default_rng(N + 1)
    rank, off, codes = geometry_reads(rng, N, [1, 2, 31, 32, 33, 63, 64, 65, 300, 1000])
    h = matrix(N)
    for H, alphabet in ((5, 7), (9, 2)):
        haps = random_haps(rng, H, N, alphabet)
        for j in range(min(H, 3)):
            i = int(rng.integers(0, len(rank)))
            haps[j, rank[i] + 1:rank[i] + 1 + np.diff(off)[i]] = codes[off[i]:off[i + 1]]
        for mm in (-1, 0, 2):
            check(h, haps, rank, off, codes, mm)


def test_long_reads():
    w = synth.scaled(synth.WORKLOADS["ont"], 5_000)
    d = synth.generate(w)
    assert d["max_k"] > 64
    haps = with_mutants(d["strains"], 20, np.random.default_rng(8), rate=0.05)
    h = matrix(w.n_snps)
    for mm in (-1, 20):
        check(h, haps, d["rank"], d["off"], d["codes"], mm)


def test_haplotypes_beyond_shared_memory():
    rng = np.random.default_rng(6)
    N = 64
    haps = random_haps(rng, 2500, N, alphabet=3)
    rank, off, codes = synth.random_packed(rng, N, 4000, 12, p_special=0.1, sort=False)
    got = check(matrix(N), haps, rank, off, codes)
    assert (got.members >= 2048).any()


def merge(parts):
    acc = {}
    for p in parts:
        for b, n in p.classes():
            acc[b] = acc.get(b, 0) + n
    return sorted(acc.items())


def test_chunked_input_equals_pieces_and_oracle():
    w = synth.scaled(synth.WORKLOADS["metagenome"], 2_200_000)
    d = synth.generate(w)
    haps = with_mutants(d["strains"], 8, np.random.default_rng(7))
    rank, off, codes = d["rank"], d["off"], d["codes"]
    assert len(rank) >= 2_000_000
    h = matrix(w.n_snps)
    whole = check(h, haps, rank, off, codes)
    cuts = [0, 123_457, 1_500_000, len(rank)]
    parts = [h.read_classes(haps, rank[a:b], off[a:b + 1], codes) for a, b in zip(cuts[:-1], cuts[1:])]
    assert whole.classes() == merge(parts)
    for f in ("assigned", "uninformative", "over_limit"):
        assert getattr(whole, f) == sum(getattr(p, f) for p in parts), f
    assert (np.diff(whole.class_off) >= 2).any()


@pytest.mark.parametrize("bits", ["0", "3"])
def test_hash_collisions(monkeypatch, bits):
    """Masked hashes: with 0 bits every tied read shares one probe chain, with 3 bits eight chains."""
    rng = np.random.default_rng(12)
    N = 120
    haps = random_haps(rng, 40, N, alphabet=2)
    rank, off, codes = synth.random_packed(rng, N, 3000, 16, p_special=0.2, sort=False)
    h = matrix(N)
    ref = check(h, haps, rank, off, codes)
    monkeypatch.setenv("HX_CLASS_HASH_BITS", bits)
    got = check(h, haps, rank, off, codes)
    assert got.classes() == ref.classes()
    assert (np.diff(got.class_off) >= 2).sum() >= 20


def test_scratch_sub_batches(monkeypatch):
    """A scratch bound of 0.01 MB (436 members) cuts the tied reads of a chunk into many sub-batches."""
    rng = np.random.default_rng(13)
    N = 200
    haps = random_haps(rng, 300, N, alphabet=2)
    rank, off, codes = synth.random_packed(rng, N, 5000, 20, p_special=0.2, sort=False)
    h = matrix(N)
    ref = check(h, haps, rank, off, codes)
    assert int((np.diff(ref.class_off) * ref.count)[np.diff(ref.class_off) >= 2].sum()) > 10 * 436
    monkeypatch.setenv("HX_CLASS_SCRATCH_MB", "0.01")
    assert check(h, haps, rank, off, codes).classes() == ref.classes()
    monkeypatch.setenv("HX_CLASS_HASH_BITS", "0")
    assert check(h, haps, rank, off, codes).classes() == ref.classes()


def test_no_reads_no_ties_all_uninformative():
    rng = np.random.default_rng(9)
    N = 30
    h = matrix(N)
    haps = random_haps(rng, 3, N)
    got = check(h, haps, np.zeros(0, np.int32), np.zeros(1, np.int64), np.zeros(0, np.uint8))
    assert len(got) == 0 and got.assigned == 0
    rank, off, codes = synth.random_packed(rng, N, 500, 10, p_special=0.1)
    got = check(h, haps[:1], rank, off, codes)                   # one haplotype: no tie
    assert (np.diff(got.class_off) == 1).all() and got.assigned > 0
    got = check(h, haps, rank, off, np.full_like(codes, 4))      # every read uninformative
    assert len(got) == 0 and got.uninformative == len(rank)
    pi = em_abundance(3, got)
    assert pi.pi.tolist() == [0.0] * 3 and pi.n_iter == 0 and pi.converged and pi.loglik == 0.0


def get_state(h):
    """hx_read_classes_get's return code (the buffers are far larger than any class set these tests leave)."""
    z64 = np.zeros(1 << 16, np.int64)
    z32 = np.zeros(1 << 16, np.int32)
    return h._lib.hx_read_classes_get(h._h, z64.ctypes.data, z32.ctypes.data, z64.ctypes.data)


def test_invalid_input_raises_and_leaves_handle_usable():
    rng = np.random.default_rng(10)
    N = 50
    h = matrix(N)
    assert get_state(h) == _lib.HX_E_STATE                      # no classes yet
    haps = random_haps(rng, 4, N)
    rank, off, codes = synth.random_packed(rng, N, 500, 20)

    def expect(code, *args):
        with pytest.raises(_lib.HanselxError) as e:
            h.read_classes(*args)
        assert e.value.code == code
        assert get_state(h) == _lib.HX_E_STATE                  # a failed call leaves no classes
        check(h, haps, rank, off, codes)                        # the handle still works

    past = np.concatenate([rank, [N - 1]]).astype(np.int32)
    expect(_lib.HX_E_READ, haps, past, np.concatenate([off, [off[-1] + 2]]), np.concatenate([codes, [0, 1]]))
    bad = codes.copy()
    bad[len(bad) // 2] = 7
    expect(_lib.HX_E_READ, haps, rank, off, bad)
    bad_hap = haps.copy()
    bad_hap[2, 3] = 7
    expect(_lib.HX_E_ARG, bad_hap, rank, off, codes)
    expect(_lib.HX_E_ARG, haps[:0], rank, off, codes)


def test_recovered_haplotypes_hiv_em():
    w = synth.WORKLOADS["hiv"]
    d = synth.generate(w)
    N = w.n_snps
    rank, off, codes = d["rank"], d["off"], d["codes"]
    h = util.load_from_packed(rank, off, codes, N, band_w=d["max_k"] - 1, device=0)
    paths, _ = h.recover_codes(h.copy(), 10)
    _, first = np.unique(paths, axis=0, return_index=True)
    haps = paths[np.sort(first)]
    band = h.band()
    got = check(h, haps, rank, off, codes)
    assert np.array_equal(h.band(), band), "read_classes changed the matrix"
    assert h.kernel_ms("classes") > 0
    for kw in ({}, {"max_iter": 7}):
        em = em_abundance(len(haps), got, **kw)
        exp = ao.em(len(haps), got.class_off, got.members, got.count, **kw)
        assert em.pi.tobytes() == np.array(exp["pi"]).tobytes()
        assert (em.n_iter, em.converged, em.loglik) == (exp["n_iter"], exp["converged"], exp["loglik"])
    # the five true strains: the EM shares against the empirical strain fractions
    strains = np.concatenate([np.full((5, 1), 6, np.uint8), d["strains"]], axis=1)
    got = check(h, strains, rank, off, codes)
    em = em_abundance(5, got)
    assert em.converged
    emp = np.bincount(d["strain_of"], minlength=5) / len(rank)
    assert np.abs(em.pi - emp).max() <= 1e-3, (em.pi, emp)


def mixture(seed=21, N=400, R=20000, k=30, p=0.8):
    """Two strains identical over sites 1..N/2 and different at every site after, drawn 80 % / 20 %: reads of 30
    sites, 1 % of their alleles changed.  Reads inside the first half tie between the strains."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 4, size=N + 1).astype(np.uint8)
    b = a.copy()
    half = N // 2
    b[half + 1:] = (a[half + 1:] + rng.integers(1, 4, size=N - half)) % 4
    haps = np.stack([a, b])
    haps[:, 0] = 6
    strain = (rng.random(R) >= p).astype(np.int64)
    rank = rng.integers(0, N - k + 1, size=R).astype(np.int32)
    off = np.arange(R + 1, dtype=np.int64) * k
    codes = haps[strain[:, None], rank[:, None] + 1 + np.arange(k)[None, :]].reshape(-1).astype(np.uint8)
    err = rng.random(len(codes)) < 0.01
    codes[err] = (codes[err] + rng.integers(1, 4, size=int(err.sum()))) % 4
    return haps, rank, off, codes, strain


def test_em_beats_equal_split_on_shared_reads():
    haps, rank, off, codes, strain = mixture()
    h = matrix(haps.shape[1] - 1)
    got = check(h, haps, rank, off, codes)
    em = em_abundance(2, got)
    truth = np.bincount(strain, minlength=2) / len(strain)
    sup = h.assign_reads(haps, rank, off, codes)
    equal = sup.share / sup.assigned
    # observed: truth 0.79355 / 0.20645; EM 0.793581 / 0.206419 (off by 3.1e-5, after 35 iterations); the equal
    # split 0.6578 / 0.3422 (off by 0.136).  Tolerances: EM within 0.005, equal split at least 0.1 off
    assert np.abs(em.pi - truth).max() <= 0.005, (em.pi, truth)
    assert np.abs(equal - truth).max() >= 0.1, (equal, truth)


# ---- command line -----------------------------------------------------------------------------------------------
def expected_abundance(bam, vcf, contig, start, end, max_paths, max_mismatch=-1):
    """gretel.abundance as the oracle flow formats it: oracle recovery, distinct paths in i_0 order, oracle classes,
    oracle EM."""
    v = bamio.process_vcf(vcf, contig, start, end)
    rank, off, codes = bamio.pack_bam(bam, contig, start, end, v)
    ho = o.load_from_packed(rank, off, codes, v["N"])
    _, PATHS = o.recover(ho, v["N"], max_paths=max_paths)
    keys = sorted(PATHS, key=lambda x: PATHS[x]["i_0"])
    haps = np.array([[REF_SYMBOLS.index(str(s)) for s in PATHS[k]["hansel_path"]] for k in keys], np.uint8)
    c = ao.classes(haps, rank, off, codes, max_mismatch)
    em = ao.em(len(keys), c["class_off"], c["members"], c["count"])
    lines = ["# %d\t%d\t%d\t%d\t%d\t%d\t%d\t%d\t%r" % (len(rank), c["assigned"], c["uninformative"], c["over_limit"],
                                                      max_mismatch, len(c["count"]), em["n_iter"], em["converged"],
                                                      em["loglik"])]
    unique, shared = [0] * len(keys), [0] * len(keys)
    for j in range(len(c["count"])):
        B = c["members"][c["class_off"][j]:c["class_off"][j + 1]]
        for m in B:
            if len(B) == 1:
                unique[m] += int(c["count"][j])
            else:
                shared[m] += int(c["count"][j])
    for j, k in enumerate(keys):
        lines.append("%d\t%d\t%d\t%.2f\t%.6f" % (PATHS[k]["i_0"], unique[j], shared[j], em["pi"][j] * c["assigned"],
                                                 em["pi"][j]))
    return lines


def run_both(tmp_path, argv, extra):
    """The same run without and with --abundance: the same outputs, plus gretel.abundance."""
    from gretel_b200 import cmd
    plain, ab = tmp_path / "plain", tmp_path / "ab"
    plain.mkdir()
    ab.mkdir()
    assert cmd.main(argv + ["-o", str(plain), "--support"] + extra) == 0
    assert cmd.main(argv + ["-o", str(ab), "--support", "--abundance"] + extra) == 0
    assert sorted(os.listdir(ab)) == ["gretel.abundance", "gretel.crumbs", "gretel.support", "out.fasta", "snp.fasta"]
    for f in ("out.fasta", "snp.fasta", "gretel.crumbs", "gretel.support"):
        assert (plain / f).read_bytes() == (ab / f).read_bytes(), f
    return open(ab / "gretel.abundance").read().split("\n")[:-1]


def test_cli_abundance_toy_bam(tmp_path, golden_dir):
    bam, vcf = os.path.join(golden_dir, "ref_test.bam"), os.path.join(golden_dir, "ref_test.vcf.gz")
    got = run_both(tmp_path, [bam, vcf, "hoot", "-s", "1", "-e", "20", "-p", "6", "--quiet"], [])
    assert got == expected_abundance(bam, vcf, "hoot", 1, 20, 6)


@pytest.mark.parametrize("max_mismatch", [-1, 1])
def test_cli_abundance_synthetic_bam(tmp_path, max_mismatch):
    bam, vcf, G = synthetic_bam(tmp_path)
    extra = ["--max-mismatch", str(max_mismatch)] if max_mismatch >= 0 else []
    got = run_both(tmp_path, [bam, vcf, "ctg", "-s", "1", "-e", str(G), "-p", "4", "--quiet", "-@", "2"], extra)
    exp = expected_abundance(bam, vcf, "ctg", 1, G, 4, max_mismatch)
    assert got == exp
    assert len(exp) >= 3

