"""Read classes and the abundance EM (DESIGN.md §4 K7) without a GPU: the numpy oracle of the classes against its
literal per-read loop and against read support, the EM on cases with a known answer, and the library's host EM
(hx_em_abundance, through ctypes) against the oracle's, bit for bit."""
import math

import numpy as np
import pytest

from gretel_b200 import _lib, synth
from gretel_b200.hansel import ReadClasses, em_abundance
from oracle import abundance_oracle as ao
from oracle import support_oracle as so

Q = 1 << 32


def random_case(seed, H=None, alphabet=None):
    rng = np.random.default_rng(seed)
    N = int(rng.integers(1, 90))
    H = int(rng.integers(1, 7)) if H is None else H
    rank, off, codes = synth.random_packed(rng, N, int(rng.integers(0, 300)), min(40, N), p_special=0.3,
                                           sort=bool(seed % 2))
    alphabet = (2 if seed % 3 == 0 else 7) if alphabet is None else alphabet
    haps = rng.integers(0, alphabet, size=(H, N + 1)).astype(np.uint8)
    return haps, rank, off, codes, [-1, 0, 1, 3][seed % 4]


def same_classes(a, b):
    for k in ("class_off", "members", "count"):
        assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), k
    for k in ("assigned", "uninformative", "over_limit"):
        assert a[k] == b[k], k


def pairs(cls):
    o = cls["class_off"]
    return [(tuple(cls["members"][o[c]:o[c + 1]].tolist()), int(cls["count"][c])) for c in range(len(cls["count"]))]


@pytest.mark.parametrize("seed", range(12))
def test_classes_match_loop(seed):
    haps, rank, off, codes, mm = random_case(seed)
    same_classes(ao.classes(haps, rank, off, codes, mm), ao.classes_loop(haps, rank, off, codes, mm))


@pytest.mark.parametrize("seed", range(3))
def test_classes_match_loop_many_haplotypes_binary(seed):
    haps, rank, off, codes, mm = random_case(100 + seed, H=300, alphabet=2)
    got = ao.classes(haps, rank, off, codes, mm)
    same_classes(got, ao.classes_loop(haps, rank, off, codes, mm))
    if got["assigned"]:
        assert (np.diff(got["class_off"]) >= 2).any()       # ties between many haplotypes are common


def class_sums(cls, H):
    """unique, shared and share_q32 per haplotype from the classes (the cross-check with K5)."""
    unique, shared, share = np.zeros(H, np.int64), np.zeros(H, np.int64), np.zeros(H, np.uint64)
    for B, n in pairs(cls):
        for h in B:
            if len(B) == 1:
                unique[h] += n
            else:
                shared[h] += n
            share[h] += np.uint64(n) * np.uint64(Q // len(B))
    return unique, shared, share


@pytest.mark.parametrize("seed", range(12))
def test_class_sums_equal_read_support(seed):
    haps, rank, off, codes, mm = random_case(seed, H=[1, 2, 5, 40][seed % 4])
    cls = ao.classes(haps, rank, off, codes, mm)
    sup = so.assign(haps, rank, off, codes, mm)
    unique, shared, share = class_sums(cls, len(haps))
    assert np.array_equal(unique, sup["unique"])
    assert np.array_equal(shared, sup["shared"])
    assert np.array_equal(share, sup["share_q32"])
    assert int(cls["count"].sum()) == cls["assigned"] == sup["assigned"]
    assert (cls["uninformative"], cls["over_limit"]) == (sup["uninformative"], sup["over_limit"])
    assert (cls["count"] >= 1).all()
    assert [b for b, _ in pairs(cls)] == sorted(b for b, _ in pairs(cls))


def csr(classes):
    """[(members, count)] -> (class_off, members, count)."""
    off = np.concatenate([[0], np.cumsum([len(b) for b, _ in classes])]).astype(np.int64)
    return off, np.array([h for b, _ in classes for h in b], np.int32), np.array([n for _, n in classes], np.int64)


def both(n_haps, classes, **kw):
    """The oracle's EM and the library's, checked bit for bit."""
    off, mem, cnt = csr(classes)
    exp = ao.em(n_haps, off, mem, cnt, **kw)
    got = em_abundance(n_haps, (off, mem, cnt), **kw)
    assert got.pi.tobytes() == np.array(exp["pi"], np.float64).tobytes()
    assert (got.n_iter, got.converged) == (exp["n_iter"], exp["converged"])
    assert np.float64(got.loglik).tobytes() == np.float64(exp["loglik"]).tobytes()
    return exp


def test_em_singletons_converge_at_iteration_two():
    counts = [7, 0, 13, 5]
    exp = both(4, [((h,), n) for h, n in enumerate(counts) if n])
    T = sum(counts)
    # iteration 1 gives count/T, iteration 2 changes nothing
    assert exp["pi"] == [n / T for n in counts]
    assert exp["n_iter"] == 2 and exp["converged"]


@pytest.mark.parametrize("a,b,c,iters", [(30, 10, 60, 51), (1, 3, 999, 5187)])
def test_em_two_haplotypes_with_shared_class(a, b, c, iters):
    """{0}:a, {1}:b, {0,1}:c: the fixed point of p = (a + c p) / (a + b + c) is a / (a + b); the error shrinks by
    c / T per iteration, so stopping at a change <= tol leaves it within tol * c / (a + b)."""
    tol = 1e-12
    exp = both(2, [((0,), a), ((0, 1), c), ((1,), b)], tol=tol)
    p = exp["pi"][0]
    assert exp["converged"] and exp["n_iter"] == iters
    assert abs(p - a / (a + b)) <= tol * c / (a + b) + 1e-15, p
    if (a, b, c) == (30, 10, 60):
        assert abs(p - 0.7499999999988) < 1e-13, p


def test_em_identical_haplotypes_keep_equal_shares():
    # haplotypes 1 and 2 are identical: every class holds both or neither
    exp = both(3, [((0,), 5), ((0, 1, 2), 40), ((1, 2), 100)])
    assert exp["pi"][1] == exp["pi"][2]
    assert exp["converged"]


def test_em_without_reads_and_without_iterations():
    exp = both(3, [])
    assert exp == {"pi": [0.0] * 3, "n_iter": 0, "converged": True, "loglik": 0.0}
    exp = both(3, [((0,), 4), ((1, 2), 2)], max_iter=0)
    assert exp["pi"] == [1.0 / 3] * 3 and exp["n_iter"] == 0 and not exp["converged"]
    assert exp["loglik"] == 4 * math.log10(1.0 / 3) + 2 * math.log10(1.0 / 3 + 1.0 / 3)


def random_classes(rng, H, n):
    sets = set()
    while len(sets) < n:
        k = int(rng.integers(1, min(H, 6) + 1))
        sets.add(tuple(sorted(rng.choice(H, size=k, replace=False).tolist())))
    return [(b, int(rng.integers(1, 1000))) for b in sorted(sets)]


@pytest.mark.parametrize("seed", range(8))
def test_library_em_equals_oracle_bit_for_bit(seed):
    rng = np.random.default_rng(seed)
    H = int(rng.integers(1, 40))
    n = int(rng.integers(1, min(60, 2 ** H - 1) + 1))
    classes = random_classes(rng, H, n)
    exp = both(H, classes)                                       # to convergence (or 10 000 iterations)
    both(H, classes, max_iter=int(rng.integers(1, 20)))          # stopped by max_iter
    both(H, classes, tol=1e-6)
    assert abs(sum(exp["pi"]) - 1.0) < 1e-9


def test_library_em_on_oracle_classes():
    haps, rank, off, codes, mm = random_case(3, H=300, alphabet=2)
    cls = ao.classes(haps, rank, off, codes, mm)
    rc = ReadClasses(cls["class_off"], cls["members"], cls["count"], cls["assigned"], cls["uninformative"],
                     cls["over_limit"])
    exp = ao.em(300, cls["class_off"], cls["members"], cls["count"], max_iter=500)
    got = em_abundance(300, rc, max_iter=500)
    assert got.pi.tobytes() == np.array(exp["pi"]).tobytes() and got.n_iter == exp["n_iter"]


@pytest.mark.parametrize("case", ["n_haps", "tol", "max_iter", "count", "member_range", "member_order",
                                  "member_repeat", "class_order", "class_repeat", "empty_class"])
def test_em_rejects_invalid_input(case):
    H, classes, kw = 3, [((0,), 2), ((0, 2), 3), ((1,), 1)], {}
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
    with pytest.raises(_lib.HanselxError) as e:
        em_abundance(H, (off, mem, cnt), **kw)
    assert e.value.code == _lib.HX_E_ARG
