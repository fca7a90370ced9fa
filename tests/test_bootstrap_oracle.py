"""The bootstrap of the abundance EM (DESIGN.md §4 K8) without a GPU: Philox4x32-10 against its known answers, the
64 x 64 -> high 64 product by 32-bit limbs, the vectorised resampler against a literal per-draw loop, the resample
against the multinomial it claims to be, and the zero-count classes that the definition leaves out of a replicate's
EM."""
import numpy as np
import pytest

from gretel_b200 import cmd
from oracle import abundance_oracle as ao
from oracle import bootstrap_oracle as bo

F = 0xFFFFFFFF
U64 = (1 << 64) - 1


@pytest.mark.parametrize("ctr, key, want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((F, F, F, F), (F, F), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert bo.philox_scalar(ctr, key) == want
    got = bo.philox(*[[c] for c in ctr], *key)
    assert tuple(int(x[0]) for x in got) == want


def test_philox_vectorised_equals_scalar():
    rng = np.random.default_rng(1)
    c = rng.integers(0, 1 << 32, size=(4, 200), dtype=np.uint64)
    k = [int(x) for x in rng.integers(0, 1 << 32, size=2)]
    got = bo.philox(*c, *k)
    for i in range(200):
        assert tuple(int(x[i]) for x in got) == bo.philox_scalar(tuple(int(v) for v in c[:, i]), tuple(k))


@pytest.mark.parametrize("T", [1, 2, 3, (1 << 31) + 1, (1 << 40) + 7, (1 << 62) + 5])
def test_mulhi(T):
    rng = np.random.default_rng(T % 1000)
    xs = [0, 1, U64, U64 - 1, 1 << 63, (1 << 32) - 1, 1 << 32] + [int(v) for v in
                                                                  rng.integers(0, 1 << 64, size=500, dtype=np.uint64)]
    got = bo.mulhi(np.array(xs, dtype=np.uint64), T)
    assert [int(v) for v in got] == [x * T >> 64 for x in xs]


def random_counts(rng, C, hi):
    return rng.integers(1, hi, size=C).astype(np.int64)


@pytest.mark.parametrize("seed", [0, 1, U64])
@pytest.mark.parametrize("case", range(6))
def test_resample_equals_per_draw_loop(seed, case):
    rng = np.random.default_rng(case)
    # T = 1, 2 (one class and two), 3, and random class sets
    count = [np.array([1], np.int64), np.array([2], np.int64), np.array([1, 1], np.int64), np.array([2, 1], np.int64),
             random_counts(rng, 40, 30), random_counts(rng, 3, 400)][case]
    T = int(count.sum())
    for b in (1, 2, 5, 1000):
        got = bo.resample(count, seed, b)
        assert np.array_equal(got, bo.resample_loop(count, seed, b)), (T, b)
        assert int(got.sum()) == T


def test_resample_chunks_do_not_matter():
    count = random_counts(np.random.default_rng(4), 30, 1000)
    assert np.array_equal(bo.resample(count, 9, 4), bo.resample(count, 9, 4, chunk_pairs=37))


def test_replicate_does_not_depend_on_the_number_of_replicates():
    count = random_counts(np.random.default_rng(5), 12, 50)
    class_off = np.arange(13, dtype=np.int64)
    members = np.arange(12, dtype=np.int32)
    a = bo.bootstrap(12, class_off, members, count, 3, 77)
    b = bo.bootstrap(12, class_off, members, count, 7, 77)
    assert np.array_equal(a["count"], b["count"][:4])
    assert a["pi"].tobytes() == b["pi"][:4].tobytes()
    assert np.array_equal(a["count"][0], count)


def test_resample_is_the_multinomial():
    count = np.array([1, 10, 100, 889], np.int64)
    T = int(count.sum())
    p = count / T
    rows = np.stack([bo.resample(count, 12345, b) for b in range(1, 4001)])
    assert (rows.sum(axis=1) == T).all()
    mean, var = rows.mean(axis=0), rows.var(axis=0, ddof=1)
    want_var = T * p * (1 - p)
    se = np.sqrt(want_var / len(rows))
    assert (np.abs(mean - T * p) <= 5 * se).all(), (mean, T * p)
    assert (np.abs(var / want_var - 1) <= 0.15).all(), (var, want_var)


def em_unfiltered(n_haps, class_off, members, count, max_iter=100):
    """K7's EM run over every class, zero counts included (what the definition does not do), in float64 numpy
    scalars so that 0/0 gives NaN instead of raising."""
    T = np.float64(sum(int(x) for x in count))
    pi = [np.float64(1.0) / n_haps] * n_haps
    with np.errstate(invalid="ignore", divide="ignore"):
        for _ in range(max_iter):
            acc = [np.float64(0.0)] * n_haps
            for c in range(len(count)):
                B = members[class_off[c]:class_off[c + 1]]
                z = np.float64(0.0)
                for h in B:
                    z += pi[h]
                for h in B:
                    acc[h] += np.float64(count[c]) * (pi[h] / z)
            pi = [a / T for a in acc]
    return pi


def test_zero_count_classes_take_no_part():
    """Haplotype 2 has one read in class {2}; a replicate that draws none of it drops the class.  Run over every
    class, the EM gives haplotype 2 pi = 0 after one iteration and then 0 * (0/0) = NaN; the definition gives finite
    values that equal K7's EM on the classes the replicate keeps."""
    class_off = np.array([0, 1, 3, 4, 5], np.int64)
    members = np.array([0, 0, 1, 1, 2], np.int32)
    count = np.array([40, 20, 39, 1], np.int64)
    T = int(count.sum())
    b = next(b for b in range(1, 100) if bo.resample(count, 3, b)[3] == 0)
    cb = bo.resample(count, 3, b)
    assert int(cb.sum()) == T and cb[3] == 0
    bad = em_unfiltered(3, class_off, members, cb)
    assert np.isnan(bad).any()
    got = bo.bootstrap(3, class_off, members, count, b, 3)
    assert np.isfinite(got["pi"][b]).all() and np.isfinite(got["loglik"][b])
    assert got["pi"][b][2] == 0.0
    o, m, n = bo.filtered(class_off, members, cb)
    exp = ao.em(3, o, m, n)
    assert got["pi"][b].tolist() == exp["pi"] and got["loglik"][b] == exp["loglik"]


def test_no_reads():
    got = bo.bootstrap(3, np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.int64), 4, 0)
    assert (got["pi"] == 0).all() and (got["n_iter"] == 0).all() and got["converged"].all()
    assert (got["loglik"] == 0).all() and got["count"].shape == (5, 0)


def test_cli_bootstrap_needs_abundance(capsys):
    with pytest.raises(SystemExit) as e:
        cmd.main(["x.bam", "x.vcf.gz", "ctg", "--bootstrap", "5"])
    assert e.value.code == 2
    assert "--bootstrap needs --abundance" in capsys.readouterr().err
