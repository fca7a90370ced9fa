"""The bootstrap of the abundance EM on the GPU (hx_em_bootstrap / Hansel.em_bootstrap, DESIGN.md §4 K8): row 0 against
the library's host EM (hx_em_abundance) bit for bit, every replicate's resampled counts against the numpy resampler of
oracle/bootstrap_oracle.py, every replicate's EM against the host EM on the classes it keeps, determinism across
batching and repeated calls, the spread of the replicates against the delta method, side effects, errors, and
gretel.bootstrap on the command line against the oracle flow."""
import os

import numpy as np
import pytest

from gretel_b200 import _lib, bamio, synth, util
from gretel_b200.gretel import boot_summary
from gretel_b200.hansel import REF_SYMBOLS, em_abundance
from oracle import abundance_oracle as ao
from oracle import bootstrap_oracle as bo
from oracle import hansel_oracle as o
from tests.test_gpu_abundance import mixture
from tests.test_gpu_read_support import matrix, random_haps, synthetic_bam, with_mutants

pytestmark = pytest.mark.gpu

U64 = (1 << 64) - 1


def csr(classes):
    """[(members, count)] -> (class_off, members, count)."""
    off = np.concatenate([[0], np.cumsum([len(b) for b, _ in classes])]).astype(np.int64)
    return off, np.array([h for b, _ in classes for h in b], np.int32), np.array([n for _, n in classes], np.int64)


def same_em(got_pi, got_it, got_conv, got_ll, exp):
    assert np.asarray(got_pi, np.float64).tobytes() == np.asarray(exp.pi, np.float64).tobytes()
    assert (int(got_it), bool(got_conv)) == (exp.n_iter, exp.converged)
    assert np.float64(got_ll).tobytes() == np.float64(exp.loglik).tobytes()


def check(h, H, cls, n_boot, seed=0, max_iter=10000, tol=1e-12, resample_rows=None):
    """em_bootstrap against the host EM: row 0 on the classes, row b on the classes with count_b >= 1; the counts of
    ``resample_rows`` (default: all) against the numpy resampler."""
    off, mem, cnt = (cls.class_off, cls.members, cls.count) if hasattr(cls, "class_off") else cls
    got = h.em_bootstrap(H, (off, mem, cnt), n_boot, seed=seed, max_iter=max_iter, tol=tol, counts=True)
    assert got.pi.shape == (n_boot + 1, H) and got.count.shape == (n_boot + 1, len(cnt))
    assert np.array_equal(got.count[0], cnt)
    assert (got.count.sum(axis=1) == int(cnt.sum())).all()
    for b in range(n_boot + 1):
        fo, fm, fc = bo.filtered(off, mem, got.count[b])
        exp = em_abundance(H, (fo, fm, fc), max_iter=max_iter, tol=tol)
        same_em(got.pi[b], got.n_iter[b], got.converged[b], got.loglik[b], exp)
    rows = range(1, n_boot + 1) if resample_rows is None else resample_rows
    for b in rows:
        assert np.array_equal(got.count[b], bo.resample(cnt, seed, b)), b
    return got


@pytest.mark.parametrize("mm", [-1, 0, 1, 3])
@pytest.mark.parametrize("H", [1, 2, 7, 33, 100, 300])
def test_grid(H, mm):
    rng = np.random.default_rng(1000 * H + 10 * (mm + 1) + 2)
    N = int(rng.integers(40, 600))
    haps = random_haps(rng, H, N, alphabet=2)
    h = matrix(N)
    rank, off, codes = synth.random_packed(rng, N, 3000, 40, p_special=0.2, sort=False)
    cls = h.read_classes(haps, rank, off, codes, max_mismatch=mm)
    check(h, H, cls, 3, seed=H + mm)


def test_grid_small_against_oracle_end_to_end():
    rng = np.random.default_rng(31)
    N = 80
    haps = random_haps(rng, 6, N, alphabet=2)
    h = matrix(N)
    rank, off, codes = synth.random_packed(rng, N, 400, 20, p_special=0.2, sort=False)
    cls = h.read_classes(haps, rank, off, codes)
    got = h.em_bootstrap(6, cls, 5, seed=5, counts=True)
    exp = bo.bootstrap(6, cls.class_off, cls.members, cls.count, 5, 5)
    assert np.array_equal(got.count, exp["count"])
    assert got.pi.tobytes() == exp["pi"].tobytes()
    assert np.array_equal(got.n_iter, exp["n_iter"]) and np.array_equal(got.converged, exp["converged"])
    assert got.loglik.tobytes() == exp["loglik"].tobytes()


def test_long_reads():
    w = synth.scaled(synth.WORKLOADS["ont"], 5_000)
    d = synth.generate(w)
    haps = with_mutants(d["strains"], 20, np.random.default_rng(8), rate=0.05)
    h = matrix(w.n_snps)
    cls = h.read_classes(haps, d["rank"], d["off"], d["codes"])
    check(h, 20, cls, 4, seed=2)


def test_haplotypes_beyond_2048():
    rng = np.random.default_rng(6)
    N = 64
    haps = random_haps(rng, 2500, N, alphabet=3)
    rank, off, codes = synth.random_packed(rng, N, 4000, 12, p_special=0.1, sort=False)
    h = matrix(N)
    cls = h.read_classes(haps, rank, off, codes)
    assert (cls.members >= 2048).any()
    check(h, 2500, cls, 2, seed=3, max_iter=300)


@pytest.mark.parametrize("a,b,c,iters", [(30, 10, 60, 51), (1, 3, 999, 5187)])
def test_anchors(a, b, c, iters):
    h = matrix(8)
    got = check(h, 2, csr([((0,), a), ((0, 1), c), ((1,), b)]), 3, seed=11)
    assert got.n_iter[0] == iters and got.converged[0]


@pytest.mark.parametrize("max_iter", [0, 7])
def test_max_iter(max_iter):
    rng = np.random.default_rng(40 + max_iter)
    classes = sorted({tuple(sorted(rng.choice(9, size=int(rng.integers(1, 4)), replace=False).tolist()))
                      for _ in range(25)})
    cls = csr([(B, int(rng.integers(1, 50))) for B in classes])
    got = check(matrix(8), 9, cls, 4, seed=1, max_iter=max_iter)
    assert (got.n_iter <= max_iter).all()
    if max_iter == 0:
        assert not got.converged.any()


def test_no_reads():
    got = matrix(8).em_bootstrap(3, csr([]), 5, counts=True)
    assert (got.pi == 0).all() and (got.n_iter == 0).all() and got.converged.all() and (got.loglik == 0).all()
    assert got.count.shape == (6, 0)


def pair_classes(H, rng):
    """Every singleton and pair of H haplotypes as a class: H (H + 1) / 2 classes in lexicographic order."""
    classes = []
    for i in range(H):
        classes.append(((i,), int(rng.integers(1, 20))))
        classes += [((i, j), int(rng.integers(1, 20))) for j in range(i + 1, H)]
    return csr(classes)


@pytest.mark.parametrize("n_boot", [1, 2, 33, 200])
@pytest.mark.parametrize("seed", [0, 1, U64])
def test_resampled_counts(n_boot, seed):
    rng = np.random.default_rng(n_boot)
    cls = pair_classes(12, rng)
    got = matrix(8).em_bootstrap(12, cls, n_boot, seed=seed, counts=True)
    for b in range(1, n_boot + 1):
        assert np.array_equal(got.count[b], bo.resample(cls[2], seed, b)), b


@pytest.mark.parametrize("count", [[1], [7], [1, 1], [1, 2], [999_000, 1, 3000, 5, 1000]])
def test_resampled_counts_edge_cases(count):
    """One class, T = 1, T = 2, and a class holding more than 99 % of the reads."""
    cls = csr([((j,), n) for j, n in enumerate(count)])
    check(matrix(8), len(count), cls, 9, seed=17)


def test_many_classes_take_the_global_paths():
    """125 250 classes: the draws search the prefix sums and count in global memory, and z does not fit in shared
    memory."""
    cls = pair_classes(500, np.random.default_rng(3))
    assert len(cls[2]) > 100_000
    check(matrix(8), 500, cls, 3, seed=U64, max_iter=40)


def test_replicate_is_independent_of_batching(monkeypatch):
    rng = np.random.default_rng(44)
    cls = pair_classes(20, rng)
    h = matrix(8)
    ref = h.em_bootstrap(20, cls, 200, seed=9, counts=True)
    again = h.em_bootstrap(20, cls, 200, seed=9, counts=True)
    for f in ("pi", "n_iter", "converged", "loglik", "count"):
        assert getattr(ref, f).tobytes() == getattr(again, f).tobytes(), f
    for b in (1, 7, 200):
        part = h.em_bootstrap(20, cls, b, seed=9, counts=True)
        assert part.pi[b].tobytes() == ref.pi[b].tobytes() and np.array_equal(part.count[b], ref.count[b])
        assert (part.n_iter[b], part.loglik[b]) == (ref.n_iter[b], ref.loglik[b])
    monkeypatch.setenv("HX_BOOT_SCRATCH_MB", "0.000001")     # one replicate per batch
    one = h.em_bootstrap(20, cls, 200, seed=9, counts=True)
    for f in ("pi", "n_iter", "converged", "loglik", "count"):
        assert getattr(ref, f).tobytes() == getattr(one, f).tobytes(), f
    check(h, 20, cls, 12, seed=9)


def test_zero_count_trap_replicates_are_finite():
    """Haplotype 2's only class holds one read: the replicates that draw none of it keep finite values equal to the
    host EM on the classes they keep."""
    cls = csr([((0,), 40), ((0, 1), 20), ((1,), 39), ((2,), 1)])
    got = check(matrix(8), 3, cls, 60, seed=3)
    trap = got.count[:, 3] == 0
    assert trap.sum() >= 5
    assert np.isfinite(got.pi).all() and np.isfinite(got.loglik).all()
    assert (got.pi[trap, 2] == 0).all()


def test_config3_full_size():
    w = synth.WORKLOADS["metagenome"]
    d = synth.generate(w)
    haps = with_mutants(d["strains"], 50, np.random.default_rng(11), rate=0.01)
    h = matrix(w.n_snps)
    cls = h.read_classes(haps, d["rank"], d["off"], d["codes"])
    assert cls.assigned >= 9_000_000
    check(h, 50, cls, 20, seed=2024, resample_rows=(1, 20))


def test_error_bars_follow_the_delta_method():
    a, b, c = 30_000, 10_000, 60_000
    h = matrix(8)
    got = h.em_bootstrap(2, csr([((0,), a), ((0, 1), c), ((1,), b)]), 1000, seed=123)
    assert got.converged.all()
    x = got.pi[1:, 0]
    s = boot_summary(x)
    p = a / (a + b)
    sd = np.sqrt(p * (1 - p) / (a + b))
    assert abs(s["boot_mean"] - p) <= 3e-4, s
    assert abs(s["boot_sd"] / sd - 1) <= 0.10, (s, sd)
    assert s["boot_lo"] <= p <= s["boot_hi"], s
    assert abs((s["boot_hi"] - s["boot_lo"]) / (2 * 1.96 * sd) - 1) <= 0.15, s


def test_mixture_intervals_contain_the_truth():
    haps, rank, off, codes, strain = mixture()
    h = matrix(haps.shape[1] - 1)
    cls = h.read_classes(haps, rank, off, codes)
    got = h.em_bootstrap(2, cls, 500, seed=5)
    truth = np.bincount(strain, minlength=2) / len(strain)
    for j in range(2):
        s = boot_summary(got.pi[1:, j])
        assert s["boot_lo"] <= truth[j] <= s["boot_hi"], (j, s, truth)


def classes_state(h):
    z64 = np.zeros(1 << 16, np.int64)
    z32 = np.zeros(1 << 16, np.int32)
    c64 = np.zeros(1 << 16, np.int64)
    rc = h._lib.hx_read_classes_get(h._h, z64.ctypes.data, z32.ctypes.data, c64.ctypes.data)
    return rc, z64.tobytes(), z32.tobytes(), c64.tobytes()


def test_side_effects_and_timers():
    w = synth.WORKLOADS["hiv"]
    d = synth.generate(w)
    rank, off, codes = d["rank"], d["off"], d["codes"]
    h = util.load_from_packed(rank, off, codes, w.n_snps, band_w=d["max_k"] - 1, device=0)
    strains = np.concatenate([np.full((5, 1), 6, np.uint8), d["strains"]], axis=1)
    cls = h.read_classes(strains, rank, off, codes)
    band, counts, state = h.band(), [h.get_counts_at(i) for i in range(0, w.n_snps + 1, 97)], classes_state(h)
    got = check(h, 5, cls, 8, seed=1)
    assert np.array_equal(h.band(), band)
    assert [h.get_counts_at(i) for i in range(0, w.n_snps + 1, 97)] == counts
    assert classes_state(h) == state
    assert h.kernel_ms("resample") > 0 and h.kernel_ms("bootstrap_em") > 0
    assert got.converged.all()


@pytest.mark.parametrize("case", ["n_haps", "tol", "max_iter", "count", "member_range", "member_order",
                                  "member_repeat", "class_order", "class_repeat", "empty_class", "n_boot"])
def test_rejects_invalid_input(case):
    H, classes, kw, n_boot = 3, [((0,), 2), ((0, 2), 3), ((1,), 1)], {}, 4
    off, mem, cnt = csr(classes)
    if case == "n_haps":
        H = 0
    elif case == "tol":
        kw["tol"] = -1e-9
    elif case == "max_iter":
        kw["max_iter"] = -1
    elif case == "count":
        cnt[1] = 0
    elif case == "member_range":
        mem[2] = 3
    elif case == "member_order":
        off, mem, cnt = csr([((0,), 2), ((2, 0), 3), ((1,), 1)])
    elif case == "member_repeat":
        off, mem, cnt = csr([((0,), 2), ((2, 2), 3)])
    elif case == "class_order":
        off, mem, cnt = csr([((0, 2), 3), ((0,), 2), ((1,), 1)])
    elif case == "class_repeat":
        off, mem, cnt = csr([((0,), 2), ((0,), 3)])
    elif case == "empty_class":
        off, mem, cnt = csr([((0,), 2), ((), 3), ((1,), 1)])
    elif case == "n_boot":
        n_boot = -1
    h = matrix(8)
    with pytest.raises(_lib.HanselxError) as e:
        h.em_bootstrap(H, (off, mem, cnt), n_boot, **kw)
    assert e.value.code == _lib.HX_E_ARG
    check(h, 3, csr(classes), 4, seed=8)                      # the handle still works


# ---- command line -----------------------------------------------------------------------------------------------
def expected_bootstrap(bam, vcf, contig, start, end, max_paths, n_boot, seed):
    """gretel.bootstrap as the oracle flow formats it: oracle recovery, distinct paths in i_0 order, oracle classes,
    the oracle bootstrap, the same numpy summaries."""
    v = bamio.process_vcf(vcf, contig, start, end)
    rank, off, codes = bamio.pack_bam(bam, contig, start, end, v)
    ho = o.load_from_packed(rank, off, codes, v["N"])
    _, PATHS = o.recover(ho, v["N"], max_paths=max_paths)
    keys = sorted(PATHS, key=lambda x: PATHS[x]["i_0"])
    haps = np.array([[REF_SYMBOLS.index(str(s)) for s in PATHS[k]["hansel_path"]] for k in keys], np.uint8)
    c = ao.classes(haps, rank, off, codes)
    em = ao.em(len(keys), c["class_off"], c["members"], c["count"])
    boot = bo.bootstrap(len(keys), c["class_off"], c["members"], c["count"], n_boot, seed)
    lines = ["# %d\t%d\t%d" % (n_boot, seed, int(boot["converged"][1:].sum()))]
    for j, k in enumerate(keys):
        s = boot_summary(boot["pi"][1:, j])
        lines.append("%d\t%.6f\t%.6f\t%.6f\t%.6f\t%.6f" % (PATHS[k]["i_0"], em["pi"][j], s["boot_mean"], s["boot_sd"],
                                                          s["boot_lo"], s["boot_hi"]))
    return lines


def run_both(tmp_path, argv):
    """The same run with --abundance, without and with --bootstrap 50 --bootstrap-seed 7: the same outputs, plus
    gretel.bootstrap."""
    from gretel_b200 import cmd
    plain, bs = tmp_path / "plain", tmp_path / "bs"
    plain.mkdir()
    bs.mkdir()
    assert cmd.main(argv + ["-o", str(plain), "--abundance"]) == 0
    assert cmd.main(argv + ["-o", str(bs), "--abundance", "--bootstrap", "50", "--bootstrap-seed", "7"]) == 0
    assert sorted(os.listdir(bs)) == ["gretel.abundance", "gretel.bootstrap", "gretel.crumbs", "out.fasta",
                                      "snp.fasta"]
    for f in ("out.fasta", "snp.fasta", "gretel.crumbs", "gretel.abundance"):
        assert (plain / f).read_bytes() == (bs / f).read_bytes(), f
    return open(bs / "gretel.bootstrap").read().split("\n")[:-1]


def test_cli_bootstrap_toy_bam(tmp_path, golden_dir):
    bam, vcf = os.path.join(golden_dir, "ref_test.bam"), os.path.join(golden_dir, "ref_test.vcf.gz")
    got = run_both(tmp_path, [bam, vcf, "hoot", "-s", "1", "-e", "20", "-p", "6", "--quiet"])
    assert got == expected_bootstrap(bam, vcf, "hoot", 1, 20, 6, 50, 7)


def test_cli_bootstrap_synthetic_bam(tmp_path):
    bam, vcf, G = synthetic_bam(tmp_path)
    got = run_both(tmp_path, [bam, vcf, "ctg", "-s", "1", "-e", str(G), "-p", "4", "--quiet", "-@", "2"])
    exp = expected_bootstrap(bam, vcf, "ctg", 1, G, 4, 50, 7)
    assert got == exp
    assert len(exp) >= 3


def test_cli_bootstrap_without_abundance_is_refused(tmp_path, golden_dir):
    from gretel_b200 import cmd
    bam, vcf = os.path.join(golden_dir, "ref_test.bam"), os.path.join(golden_dir, "ref_test.vcf.gz")
    with pytest.raises(SystemExit) as e:
        cmd.main([bam, vcf, "hoot", "-s", "1", "-e", "20", "-o", str(tmp_path), "--bootstrap", "5"])
    assert e.value.code == 2
